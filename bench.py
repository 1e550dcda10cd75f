#!/usr/bin/env python3
"""bench.py -- headline benchmark of the NAVTEX receive chain (BASELINE.json metric:
"IQ Msamples/s through FIR cascade + FSK demod at 1-8 B200; % HBM roofline").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A step = one pass of the whole hot path (fused FIR cascade -> demod / bit-sync -> SITOR-B state
machine -> host message assembly) over one block of BASELINE.json configs[1]: 1024 synthetic IQ
streams per GPU (distinct SITOR-B bulletins, start times, channels and SNRs) x 10.28 s at 252 kS/s,
resident in HBM (21 GB per GPU: far larger than the 126 MB L2, so nothing is cache-warm between
steps).  Streams are independent: N GPUs = N x 1024 streams, no collective on the data path
(weak scaling); the only cross-rank traffic is the barrier, the max-over-ranks timing, the sums of the
check counters and the final host gather of the decoded messages.

value  = samples processed by all ranks / max-over-ranks device time (CUDA events on the engine stream).
e2e    = same metric through nvx_engine_push_host_s16 (the reference's own int16 sample format) with
         pinned HOST buffers: the same captures pushed as consecutive 1.03 s blocks; H2D copy, int16->float
         conversion, all kernels, event download and host message assembly inside the timed region, the
         decoded bulletins checked against what was transmitted, and -- beside it -- the rate of a bare pinned
         cudaMemcpyAsync of the same bytes on all ranks at once (the PCIe / host ceiling of this box at this N).
The one JSON line also carries, each with its own check (and every rank verifies its OWN streams; the counts are summed):
  check.oracle_parity  same-run parity of 64 of the workload's streams against the UNMODIFIED reference (oracle/_ref/ref_chain)
  int16_input          the same captures resident as int16 (fused-ingest kernel variant, FP32-bound)
  config4              BASELINE.json configs[3]: 8192 streams per GPU (65536 at --gpus 8) of traffic generated per block
  config5              BASELINE.json configs[4]: the long-tap stress (255-tap filters, tensor-core stages)
  cpu_baseline         the reference's CPU chain on this box's host cores (one pinned core, and all cores)
--impl reference times the reference's own CPU chain (oracle/_ref/ref_chain_timing, built unmodified from
the reference sources, no taps) on all host cores on a bounded sample of the same workload.
"""
from __future__ import annotations

import argparse
import collections
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

STREAMS_PER_GPU = 1024
SUPER_PER_BLOCK = 9250              # 900 Hz outputs per stream per step -> n = 2,590,000 samples (10.28 s)
BLOCK = SUPER_PER_BLOCK * 280
E2E_CHUNKS = 10                     # the e2e arm pushes the same captures as 10 consecutive host blocks ...
E2E_BLOCK = BLOCK // E2E_CHUNKS     # ... of 259,000 samples (1.03 s) per stream: 1.06 GB of int16 per step
BYTES_PER_SAMPLE = 8.0 + 16.0 / 280 # algorithmic HBM bytes per input IQ sample (SURVEY.md 8d): float2 in, 2 x float2 per 280 out
REF_CHAIN = os.path.join(ROOT, "oracle", "_ref", "ref_chain")                 # with the --wrap stage taps: parity
REF_CHAIN_TIMING = os.path.join(ROOT, "oracle", "_ref", "ref_chain_timing")   # same objects, no interposers: timing
PARITY_STREAMS = 64
C4_STREAMS = 8192
C4_BLOCK = 1125 * 280               # 1.25 s per stream per block: 20.6 GB of float2 per GPU


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f)
    except Exception:
        return {}


def measured_peak():
    p = measured_peaks()
    if "hbm_gbs" in p:
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic():
    """DRAM bytes per launch of the fused kernel from the committed ncu --set full capture (a run under ncu is never a bench
    value, so this cannot be measured live): profiles/cascade_traffic.json says from which command, commit and date."""
    try:
        with open(os.path.join(ROOT, "profiles", "cascade_traffic.json")) as f:
            return json.load(f)
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def wait_first(self, timeout=5.0):
        """nvidia-smi needs a moment to start: do not enter a timed region before its first sample has arrived."""
        t0 = time.time()
        while self.proc and not self.rows and time.time() - t0 < timeout:
            time.sleep(0.02)

    def window(self, t0, t1):
        """Clock record of [t0, t1] (the sampler keeps running: one process serves every timed region of the run)."""
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.06)
        rows = list(self.rows)
        # samples inside the timed region; a region shorter than the sampling period falls back to the samples taken
        # while the warm-up steps (same kernels, same load) were running just before it
        inside = [r for ts, r in rows if t0 <= ts <= t1 + 0.03 and len(r) >= 7]
        how = "inside the timed region"
        if not inside:
            inside = [r for ts, r in rows if t0 - 0.5 <= ts <= t1 + 0.1 and len(r) >= 7]
            how = "timed region shorter than the sampling period: samples within 0.5 s before it (warm-up steps, same load)"
        if not inside:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [nm for k, nm in enumerate(names) if any(r[3 + k].lower().startswith("active") for r in inside)]

        def num(x):
            try:
                return float(x)
            except ValueError:
                return None
        sm = [num(r[0]) for r in inside if num(r[0]) is not None]
        pw = [num(r[2]) for r in inside if num(r[2]) is not None]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": num(inside[0][1]), "power_w_max": max(pw) if pw else None,
                "samples": len(inside), "sampled": how, "reasons": reasons}

    def close(self):
        if self.proc:
            self.proc.terminate()


def bind_cpus(local, world):
    """Give every rank its own CPUs (and so its pinned host buffers' first touch): the CPUs of the NUMA node its GPU hangs off
    when sysfs shows one, split evenly over the ranks that share it; otherwise a round-robin split of the CPUs this process may
    run on.  Matters for the e2e arm at N > 1, where every GPU pulls 55 GB/s out of host memory."""
    info = {"numa_node": None}
    try:
        cpus = sorted(os.sched_getaffinity(0))
        try:
            bdf = subprocess.run(["nvidia-smi", "-i", str(local), "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                                 capture_output=True, text=True, timeout=20).stdout.strip().lower()
            if bdf.startswith("0000"):
                bdf = bdf[4:]                  # nvidia-smi prints an 8-digit domain, sysfs uses 4
            node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read())
            if node >= 0:
                node_cpus = set()
                for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
                    lo, _, hi = part.partition("-")
                    node_cpus.update(range(int(lo), int(hi or lo) + 1))
                if node_cpus & set(cpus):
                    cpus = sorted(node_cpus & set(cpus))
                    info["numa_node"] = node
        except Exception:
            pass
        per = max(1, len(cpus) // max(1, world))
        mine = cpus[(local * per) % len(cpus):][:per] or cpus
        os.sched_setaffinity(0, mine)
        info["cpus"] = f"{mine[0]}-{mine[-1]}" if len(mine) > 1 else str(mine[0])
        info["n_cpus"] = len(mine)
    except Exception as ex:       # affinity is a tuning aid, never a reason to fail
        info["error"] = str(ex)
    return info


def make_bulletins(np, synth, S, rank, seed, fit_samples, n_lines, words, n_phasing, n_tail, seconds=None):
    """S distinct bulletins for this rank: bit strings, channel, start time, amplitude, noise -- and what must come out."""
    rng = np.random.default_rng(seed + rank)
    bits, off, start, amp, sigma, expect = [], [], [], [], [], []
    for s in range(S):
        while True:      # bulletins short enough to fit the capture together with their start delay
            text, bbbb = synth.random_message(rng, n_lines=n_lines, words_per_line=words)
            b = synth.message_bits(text, n_phasing=n_phasing, n_tail=n_tail)
            if len(b) * 2520 + 0.6 * 252000 < fit_samples:
                break
        bits.append(b)
        ch = s % 2
        off.append(14000.0 if ch == 0 else -14000.0)
        if seconds is None:
            start.append(0.05 + 0.4 * rng.random())
        else:
            start.append(0.3 + max(0.0, seconds - len(b) / 100.0 - 1.2) * rng.random())
        amp.append(3000.0 + 6000.0 * rng.random())
        sigma.append(amp[-1] * 10 ** (rng.uniform(-6.0, 14.0) / 20) / np.sqrt(2))     # full-band SNR -14 .. +6 dB
        expect.append((s + rank * S, 518 if ch == 0 else 490, bbbb, text))
    return bits, off, start, amp, sigma, expect


def build_workload(torch, device, rank):
    """1024 distinct synthetic captures for this rank, generated on the device (untimed)."""
    import numpy as np
    from navtex_b200 import engine, synth

    S = STREAMS_PER_GPU
    bits, off, start, amp, sigma, expect = make_bulletins(np, synth, S, rank, 518490, BLOCK, 1, 3, 18, 5)
    x = torch.empty((S, BLOCK, 2), dtype=torch.float32, device=device)
    engine.synth_fill_device(device.index, x.data_ptr(), S, 0, BLOCK, bits, off, start, amp, sigma, seed=518490 + rank)
    return x, expect


def count_exact(msgs, expect):
    got = collections.Counter((m[0], m[1], m[2], m[3]) for m in msgs)
    return sum(1 for e in expect if got.get(e, 0) > 0), got


# ------------------------------------------------------------------------------------------- CPU reference chain
def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def ref_binary():
    for p in (REF_CHAIN_TIMING, REF_CHAIN):
        if os.path.exists(p):
            return p
    return None


RATES = []      # Msamples/s of every timed wave-pass of the last run_reference_cpu calls (the host is a noisy VM: spread matters)


def run_reference_cpu(samples_i16, passes_warm, passes_timed, cores, pin_core=None):
    """Time the unmodified reference chain: one process (= one stream: its state is global) per core, `cores` at a time,
    until every stream of the sample has been through; passes back to back on the same in-memory capture.  A pass of a wave
    ends when its slowest process finishes it.  Returns (samples/s, mean seconds per wave-pass, samples per stream)."""
    import numpy as np

    exe = ref_binary()
    n = samples_i16[0].size // 2
    wave_s, total = 0.0, 0
    with tempfile.TemporaryDirectory() as td:
        paths = []
        for k, iq in enumerate(samples_i16):
            p = os.path.join(td, f"s{k}.s16")
            np.ascontiguousarray(iq, dtype=np.int16).tofile(p)
            paths.append(p)
        for w0 in range(0, len(paths), cores):
            wave = paths[w0:w0 + cores]

            def pre(k):
                if pin_core is None:
                    return None
                return lambda: os.sched_setaffinity(0, {pin_core})
            procs = [subprocess.Popen([exe, "--s16", p, "--passes", str(passes_warm + passes_timed)], stdout=subprocess.DEVNULL,
                                      stderr=subprocess.PIPE, text=True, preexec_fn=pre(k)) for k, p in enumerate(wave)]
            outs = [p.communicate()[1] for p in procs]
            per_pass = [json.loads(o.strip().splitlines()[-1])["pass_s"][passes_warm:] for o in outs]
            wave_pass = [max(pp[k] for pp in per_pass) for k in range(passes_timed)]
            wave_s += sum(wave_pass)
            total += len(wave) * n * passes_timed
            RATES.extend(len(wave) * n / t / 1e6 for t in wave_pass)
    waves = (len(paths) + cores - 1) // cores
    return total / wave_s, wave_s / (waves * passes_timed), n


def cpu_reference_figures(sample, warm, timed):
    """The reference CPU chain on this box: (i) one process pinned to one core, (ii) one process per host core.
    sample = list of int16 captures (>= 64 of the workload's streams, first seconds of each)."""
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    if ref_binary():
        one = sorted(os.sched_getaffinity(0))[0]
        sps1, _, n = run_reference_cpu(sample[:4], 1, timed, 1, pin_core=one)
        del RATES[:]
        sps, step_s, n = run_reference_cpu(sample, warm, timed, cores)
        kind, binary = "reference", os.path.relpath(ref_binary(), ROOT)
    else:   # the compiled reference did not travel: time the C port instead (single thread)
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import oracle_lib as ol
        t0 = time.time()
        for k in range(4):
            ol.run_oracle(sample[k % len(sample)], record_taps=False)
        n = sample[0].size // 2
        sps1 = sps = 4 * n / (time.time() - t0)
        step_s, cores, kind, binary = n / sps, 1, "port", "oracle/libnavtex_oracle.so"
    desc = (f"first {n / 252000:.1f} s of {len(sample)} of the workload's streams; one {os.path.basename(binary)} process per core, "
            f"{cores} at a time, {warm} warm-up + {timed} timed passes each, a wave-pass ends with its slowest process")
    return {"value": sps / 1e6, "unit": "Msamples/s", "cores": cores, "kind": kind, "sample": desc,
            "one_core_pinned_msamples_per_s": sps1 / 1e6, "per_core_msamples_per_s": sps / 1e6 / max(1, cores),
            "realtime_streams": sps / 252000.0, "nproc": os.cpu_count(), "cpu_model": cpu_model(), "binary": binary,
            "streams_in_sample": len(sample), "samples_per_stream": n,
            "wave_pass_msamples_per_s": {"min": min(RATES), "median": statistics.median(RATES), "max": max(RATES), "n": len(RATES)} if RATES else None}, step_s


def reference_sample(np, synth, n_streams, seconds):
    rng = np.random.default_rng(518490)
    streams = []
    for s in range(n_streams):
        text, _ = synth.random_message(rng, n_lines=1, words_per_line=2)
        em = synth.Emission(text, 14000.0 if s % 2 == 0 else -14000.0, start_s=0.1, n_phasing=12, n_tail=4)
        streams.append(synth.quantise_s16(synth.fsk_iq([em], seconds, snr_db=float(rng.uniform(-14, 6)), seed=s)))
    return streams


def impl_reference(args, rank, world):
    if rank != 0:
        return
    import numpy as np
    from navtex_b200 import synth

    sample = reference_sample(np, synth, 64, 4.0)        # bounded sample: 4 s of each of 64 streams of the workload's kind
    cpu, step_s = cpu_reference_figures(sample, args.warmup, args.steps)
    val = cpu["value"]
    line = {
        "impl": "reference", "metric": "iq_msamples_per_s", "value": val, "unit": "Msamples/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": step_s * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "configs[1]: 1024 synthetic IQ streams/GPU, fused FIR cascade + FSK demod + bit-sync + SITOR-B (CPU chain on host cores, bounded sample)",
                   "streams_per_gpu": STREAMS_PER_GPU, "sample": cpu["sample"]},
        "cpu_baseline": cpu,
        "e2e": {"value": val, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "realtime_streams": val / 0.252,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------- legs of the GPU arm
class Ctx:
    pass


def allreduce_max(c, v):
    t = c.torch.tensor([v], dtype=c.torch.float64, device=c.device)
    if c.world > 1:
        c.dist.all_reduce(t, op=c.dist.ReduceOp.MAX)
    return float(t.item())


def allreduce_sum(c, values):
    t = c.torch.tensor(list(values), dtype=c.torch.float64, device=c.device)
    if c.world > 1:
        c.dist.all_reduce(t, op=c.dist.ReduceOp.SUM)
    return [int(round(v)) for v in t.tolist()]


def verify_all_ranks(c, msgs, expect, steps):
    """Every rank checks ITS OWN bulletins (how many of the expected ones came out verbatim; whether the multiset of what came
    out is exactly `steps` copies of each expected one: nothing missing, nothing extra, nothing garbled); rank 0 additionally
    gathers every rank's messages and expectations -- the job's only cross-rank data exchange, untimed -- and compares the
    gathered multiset with the union.  Returns (exact count, multiset flag, rank-0 check record)."""
    from navtex_b200 import sharding

    decoded_ok, got = count_exact(msgs, expect)
    multiset_ok = int(got == collections.Counter({e: steps for e in expect}))
    check = {"bulletins_expected_per_step_per_gpu": len(expect), "decoded_exact_rank0": decoded_ok}
    merged = sharding.gather_messages(msgs)
    all_expect = [None] * c.world if c.rank == 0 else None
    if c.world > 1:
        c.dist.gather_object(expect, all_expect, dst=0)
    else:
        all_expect = [expect]
    if c.rank == 0:
        want = collections.Counter({e: steps for ex in all_expect for e in ex})
        have = collections.Counter((m[0], m[1], m[2], m[3]) for m in merged)
        check["messages_gathered_all_ranks"] = len(merged)
        check["gathered_multiset_equals_union_of_expected"] = bool(want == have)
    return decoded_ok, multiset_ok, check


def timed_pushes(c, eng, ptr, n, steps, warmup, s16=False, reset=False):
    """warmup untimed pushes, then exactly `steps` pushes of the resident block bracketed by barrier + synchronize; device time
    by CUDA events on the engine's stream, max over ranks.  Returns (ms, stats, messages of the timed pushes, clocks, spans)."""
    torch = c.torch
    es = torch.cuda.ExternalStream(eng.stream, device=c.device)
    for _ in range(warmup):
        eng.push_device(ptr, n, s16=s16)
    eng.poll_messages()
    if reset:
        eng.reset()
    eng.enable_timing(1)            # two event records per block around the fused FIR kernel, nothing else
    eng.stats()
    if c.sampler:
        c.sampler.wait_first()
    c.barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_wall0 = time.time()
    ev0.record(es)
    for _ in range(steps):
        eng.push_device(ptr, n, s16=s16)
    eng.sync()
    ev1.record(es)
    c.barrier()
    t_wall1 = time.time()
    clocks = c.sampler.window(t_wall0, t_wall1) if c.sampler else None
    ms = allreduce_max(c, ev0.elapsed_time(ev1))
    spans = eng.cascade_spans()
    st = eng.stats()
    msgs = eng.poll_messages()
    eng.enable_timing(0)
    return ms, st, msgs, clocks, spans


DUMP_Y3_STREAMS = 128       # 18.9 MB of y3: the whole [1024][2][9250] complex64 block would be 152 MB


def dump_outputs(eng, out_dir):
    """What a caller of the timed path receives after its last step, as float32 .npy files, so that two builds can be compared
    output for output: y3.npy [K][channel][900 Hz sample][re, im] of a fixed, seeded sample of K streams (their indices in
    y3_streams.npy) and events.npy [stream][channel][byte] of every stream's decoded event bytes, padded with -1."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    pick = np.sort(np.random.default_rng(0).choice(eng.S, size=min(DUMP_Y3_STREAMS, eng.S), replace=False))
    y3 = np.ascontiguousarray(eng.read_y3()[pick])
    np.save(os.path.join(out_dir, "y3.npy"), y3.view(np.float32).reshape(*y3.shape, 2))
    np.save(os.path.join(out_dir, "y3_streams.npy"), pick.astype(np.float32))
    ev = [[eng.read_events(s, ch) for ch in range(eng.C)] for s in range(eng.S)]
    out = np.full((eng.S, eng.C, max(1, max(len(e) for row in ev for e in row))), -1.0, dtype=np.float32)
    for s, row in enumerate(ev):
        for ch, e in enumerate(row):
            out[s, ch, :len(e)] = np.frombuffer(e, dtype=np.uint8)
    np.save(os.path.join(out_dir, "events.npy"), out)


def span_stats(spans):
    if len(spans) == 0:
        return {"kernel_ms_min": None, "kernel_ms_median": None, "kernel_ms_max": None}
    return {"kernel_ms_min": float(min(spans)), "kernel_ms_median": float(statistics.median(map(float, spans))), "kernel_ms_max": float(max(spans))}


def leg_oracle_parity(c, x, expect, n_streams=PARITY_STREAMS):
    """Same-run parity (BASELINE.md 4-5): PARITY_STREAMS of this rank's streams, the full 10.28 s, through the UNMODIFIED
    reference (oracle/_ref/ref_chain --out: stage taps by ld --wrap) on the host cores, against one more pass of the GPU chain
    over the resident block with the bit taps switched on.  Rank 0 only.  Messages, events-to-text and bit decisions of the
    occupied channel exact; 900 Hz samples and discriminator sums within 1e-5 / 5e-5 (tests/parity.py says of what)."""
    import numpy as np
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as ol
    import parity
    from navtex_b200 import engine

    S = STREAMS_PER_GPU
    eng = engine.Engine(S, BLOCK, device=c.local, first_stream_id=c.rank * S, keep_bits=True)
    eng.push_device(x.data_ptr(), BLOCK)
    msgs = eng.poll_messages()
    y3 = eng.read_y3()
    n_streams = max(1, min(S, n_streams))
    pick = list(range(0, S, S // n_streams))[:n_streams]
    caps = [x[s].round().to(c.torch.int16).cpu().numpy().reshape(-1) for s in pick]
    use_ref = ol.have_ref()
    t0 = time.time()
    if use_ref:
        from concurrent.futures import ThreadPoolExecutor
        with ThreadPoolExecutor(max_workers=len(os.sched_getaffinity(0))) as pool:       # one ref_chain process per stream
            refs = list(pool.map(lambda iq: ol.run_ref(iq), caps))
    else:
        refs = [ol.run_oracle(iq) for iq in caps]
    cpu_s = time.time() - t0
    cmps, occ, msg_ok = [], [], 0
    by_stream = collections.defaultdict(list)
    for m in msgs:
        by_stream[m[0]].append((m[1], m[2], m[3]))
    for s, r in zip(pick, refs):
        bits, disc = {}, {}
        for ch in (0, 1):
            bits[ch], disc[ch] = eng.read_bits(s, ch)
        tags = {parity.CHANNELS[s % 2]}
        cmps.append(parity.compare_stream(y3[s], bits, disc, r, tags))
        occ.append(tags)
        msg_ok += int(by_stream.get(s + c.rank * S, []) == r.messages and len(r.messages) == 1)
    eng.close()
    out = parity.summarise(cmps, occ)
    out.update({"against": "oracle/_ref/ref_chain (unmodified reference sources, FP64)" if use_ref else "oracle/libnavtex_oracle.so (C restatement; the compiled reference did not travel)",
                "samples_per_stream": BLOCK, "messages_exact": msg_ok, "cpu_seconds": cpu_s,
                "bars": {"y3_rel": parity.REL_TOL, "disc_rel": 5 * parity.REL_TOL, "bits_occupied": "identical", "messages": "identical"}})
    out["pass"] = bool(out["y3_max_rel_pair_peak"] <= parity.REL_TOL and (out["y3_max_rel_own_rms_occupied"] or 0) <= parity.REL_TOL and
                       out["bit_mismatches_occupied"] == 0 and msg_ok == len(pick) and (out["disc_max_rel_occupied"] or 0) <= 5 * parity.REL_TOL)
    return out


def leg_e2e(c, x, expect, args):
    """End to end through the host-buffer C ABI: the same 1024 captures, as the reference's int16 samples in page-locked host
    memory (nvx_pinned_alloc), pushed as consecutive 1.03 s blocks (step k pushes chunk k mod 10; after the tenth the captures
    start over, like a new emission).  Then the ceiling: a bare pinned cudaMemcpyAsync of the same chunks, all ranks at once."""
    import numpy as np
    from navtex_b200 import engine

    torch, S, ne = c.torch, STREAMS_PER_GPU, E2E_BLOCK
    assert ne % 280 == 0 and ne * E2E_CHUNKS == BLOCK
    pinned = engine.PinnedBuffer((E2E_CHUNKS, S, ne, 2), np.int16, write_combined=args.pinned == "wc")
    host = torch.from_numpy(pinned.array)
    for k in range(E2E_CHUNKS):
        host[k].copy_(x[:, k * ne:(k + 1) * ne].round().to(torch.int16))
    chunk_ptr = [pinned.ptr + k * S * ne * 4 for k in range(E2E_CHUNKS)]
    eng = engine.Engine(S, ne, device=c.local, first_stream_id=c.rank * S)
    es = torch.cuda.ExternalStream(eng.stream, device=c.device)
    warm = E2E_CHUNKS * max(1, (max(3, args.warmup) + E2E_CHUNKS - 1) // E2E_CHUNKS)     # whole captures, so step 0 starts one
    for k in range(warm):
        eng.push_host_ptr(chunk_ptr[k % E2E_CHUNKS], ne, s16=True)
        eng.poll_messages()
    c.barrier()
    a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    tw0 = time.time()
    a0.record(es)
    msgs = []
    for k in range(args.steps):
        eng.push_host_ptr(chunk_ptr[k % E2E_CHUNKS], ne, s16=True)
        # every block's events are downloaded (D2H) and assembled on the host as part of its push; collect what has
        # completed so far without stalling the copy / compute pipeline
        msgs += eng.poll_messages(wait=False)
    msgs += eng.poll_messages()                               # drain: the last blocks' results, inside the timed region
    a1.record(es)
    c.barrier()
    wall = time.time() - tw0
    sec = allreduce_max(c, max(a0.elapsed_time(a1) * 1e-3, wall))
    eng.close()
    # ---- ceiling: the same bytes, nothing but the copies, every rank at the same time
    scratch = torch.empty((S, ne, 2), dtype=torch.int16, device=c.device)
    cs = torch.cuda.Stream(device=c.device)
    n_copy = max(10, min(args.steps, 40))
    bytes_chunk = S * ne * 4

    def copies(n):          # tensor.copy_ from page-locked memory = one cudaMemcpyAsync per chunk on stream cs
        with torch.cuda.stream(cs):
            for k in range(n):
                scratch.copy_(host[k % E2E_CHUNKS], non_blocking=True)
    copies(3)
    cs.synchronize()
    c.barrier()
    b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    b0.record(cs)
    copies(n_copy)
    b1.record(cs)
    cs.synchronize()
    c.barrier()
    copy_s = allreduce_max(c, b0.elapsed_time(b1) * 1e-3)
    ceiling = c.world * bytes_chunk * n_copy / copy_s / 1e9
    del scratch, host
    pinned.close()
    value = c.world * S * ne * args.steps / sec / 1e6
    gbs = c.world * bytes_chunk * args.steps / sec / 1e9
    ev_cap = 2 * (ne // 280 // 63 + 2) + 8
    expected = len(expect) * (args.steps // E2E_CHUNKS)
    expect_set = set(expect)
    exact = sum(1 for m in msgs if (m[0], m[1], m[2], m[3]) in expect_set)
    e2e = {"value": value, "unit": "Msamples/s", "h2d_bytes_per_step": bytes_chunk, "d2h_bytes_per_step": 2 * S * (ev_cap + 4),
           "input": f"int16 IQ in page-locked host memory ({args.pinned}), [{S} streams][{ne} samples] per step per GPU, consecutive blocks of the same captures",
           "ms_per_step": sec * 1e3 / args.steps, "h2d_gbs": gbs,
           "h2d_ceiling_gbs": ceiling, "frac_of_ceiling": (gbs / ceiling) if ceiling else None,
           "ceiling": f"bare pinned cudaMemcpyAsync of the same chunks, {n_copy} copies per rank, all {c.world} ranks at once, max over ranks",
           "cpu_binding": c.cpus}
    return e2e, len(msgs), exact, expected


def leg_config4(c, seconds, warm_blocks=1, standalone=False):
    """BASELINE.json configs[3]: 8192 streams per GPU (65536 over 8 GPUs) of traffic, too large to be resident (124 GB per 8 s as
    float2): generated on the device block by block (counter-based generator keyed by (seed, stream, absolute sample): any
    block of any stream is reproducible) and decoded through the carried state.  Generation is untimed; every block's span
    covers ALL of its kernels and its event download (nvx_engine_fence puts the span's end behind the demod stream), so no
    overlap between a block's sequential demod kernels and the next block is credited: a lower bound on the pipelined rate."""
    import numpy as np
    from navtex_b200 import engine, sharding, synth

    torch, S, block = c.torch, C4_STREAMS, C4_BLOCK
    n_blocks = max(1, int(round(seconds * 252000 / block)))
    seconds = n_blocks * block / 252000
    if standalone:   # the full 60 s: two-line bulletins anywhere in the minute
        bits, off, start, amp, sigma, expect = make_bulletins(np, synth, S, c.rank, 65536, int(seconds * 252000), 2, 4, 30, 6, seconds=seconds)
    else:            # the folded short pass: bulletins that complete inside `seconds`
        bits, off, start, amp, sigma, expect = make_bulletins(np, synth, S, c.rank, 65536, int(seconds * 252000), 1, 3, 18, 5, seconds=seconds)
    bufs = [torch.empty((S, block, 2), dtype=torch.float32, device=c.device) for _ in range(2)]
    eng = engine.Engine(S, block, device=c.local, first_stream_id=c.rank * S)
    es = torch.cuda.ExternalStream(eng.stream, device=c.device)

    def generate(k):
        engine.synth_fill_device(c.local, bufs[k % 2].data_ptr(), S, k * block, block, bits, off, start, amp, sigma,
                                 seed=65536 + c.rank, cuda_stream=eng.stream)

    generate(0)
    for _ in range(warm_blocks):
        eng.push_device(bufs[0].data_ptr(), block)       # warm-up (engine reset afterwards)
    eng.poll_messages()
    eng.reset()
    eng.enable_timing(1)
    eng.stats()
    if c.sampler:
        c.sampler.wait_first()
    c.barrier()
    spans = []
    t_wall0 = time.time()
    for k in range(n_blocks):
        generate(k)                                       # host-synchronous: the engine's streams are idle when it returns
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(es)
        eng.push_device(bufs[k % 2].data_ptr(), block)
        eng.fence()                                       # main stream waits for the block's demod stream work ...
        e1.record(es)                                     # ... so the span ends after its last kernel and its event download
        spans.append((e0, e1))
    eng.sync()
    torch.cuda.synchronize()
    c.barrier()
    t_wall1 = time.time()
    clocks = c.sampler.window(t_wall0, t_wall1) if c.sampler else None
    dec_ms = allreduce_max(c, sum(a.elapsed_time(b) for a, b in spans))
    casc = eng.cascade_spans()
    st = eng.stats()
    msgs = eng.poll_messages()
    ok, _ = count_exact(msgs, expect)
    ok_all, exp_all, n_all = allreduce_sum(c, [ok, len(expect), len(msgs)])
    merged = sharding.gather_messages(msgs) if standalone else None
    eng.close()
    del bufs
    torch.cuda.empty_cache()
    total = c.world * S * block * n_blocks
    peak, peak_src = measured_peak()
    casc_ms = st.cascade_ms / max(1, st.cascade_launches)
    rec = {
        "value": total / (dec_ms * 1e-3) / 1e6, "unit": "Msamples/s", "steps": n_blocks, "ms_per_step": dec_ms / n_blocks,
        "workload": "configs[3]: %d streams per GPU (%d in all) x %.2f s of traffic, generated on the device per 1.25 s block (20.6 GB float2 per GPU, "
                    "regenerated every block: nothing cache-warm)" % (S, S * c.world, seconds),
        "streams_total": S * c.world, "seconds_of_traffic": seconds,
        "timing": {"decode_ms": dec_ms, "wall_ms_including_generation": (t_wall1 - t_wall0) * 1e3,
                   "how": "sum over blocks of the CUDA-event span push -> fence (all kernels of the block incl. its sequential demod kernels and event "
                          "download; generator untimed), max over ranks; blocks do not overlap, so a lower bound on the pipelined rate"},
        "realtime_streams": total / (dec_ms * 1e-3) / 252000,
        "roofline": {"bound": "hbm", "achieved": S * block * BYTES_PER_SAMPLE / (casc_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                     "frac": S * block * BYTES_PER_SAMPLE / (casc_ms * 1e-3) / 1e9 / peak, "peak_source": peak_src,
                     "kernel": "nvx::fir_cascade_kernel<true,false,false,0>", "kernel_ms": casc_ms, **span_stats(casc)},
        "gpu_launches": int(st.cascade_launches + st.demod_launches + st.aux_launches), "clocks": clocks,
        "check": {"bulletins_complete_in_capture_all_ranks": exp_all, "decoded_exact_all_ranks": ok_all, "messages_total_all_ranks": n_all},
    }
    if merged is not None:
        rec["check"]["messages_gathered_all_ranks"] = len(merged)
    return rec


def leg_config5(c, x, expect, taps_n, steps, warmup):
    """BASELINE.json configs[4]: long-tap FIR stress.  The default workload's 1024 captures per GPU, resident in HBM, through
    taps_n-tap Kaiser designs in all three stages (steeper than fir1cpp.C:8 / fir2cpp.C:22 / fir3cpp.h:16): stages 1 and 2 run
    on the tensor cores (fir_long_tc.cu), stage 3 and the demod chain as usual; every bulletin is checked."""
    from scipy import signal
    from navtex_b200 import engine

    S, T = STREAMS_PER_GPU, taps_n
    taps = (signal.firwin(T, 20000, window=("kaiser", 8.0), fs=252000), signal.firwin(T, 2000, window=("kaiser", 8.0), fs=63000),
            signal.firwin(T, 250, window=("kaiser", 7.0), fs=9000))
    eng = engine.Engine(S, BLOCK, device=c.local, first_stream_id=c.rank * S, taps=taps)
    note = eng.L.nvx_last_error().decode()
    ms, st, msgs, clocks, spans = timed_pushes(c, eng, x.data_ptr(), BLOCK, steps, warmup, reset=True)
    ok, _ = count_exact(msgs, expect)       # the first pass decodes every bulletin; later passes continue the same streams
    ok_all, exp_all, n_all = allreduce_sum(c, [ok, len(expect), len(msgs)])
    eng.close()
    total = c.world * S * BLOCK * steps
    flop = 4.0 * T * (1 / 4 + 2 / 28 + 2 / 280) + 6 / 4          # per input sample: real FMAs x 2 per complex-by-real tap, + the mix
    fir_ms = st.cascade_ms / max(1, st.cascade_launches)         # the three stage kernels of one block (CUDA events)
    p = measured_peaks()
    if "bf16_tflops" in p:
        peak, peak_src = float(p["bf16_tflops"]) / 2, "measured dense bf16 TF/s (MEASURED_PEAKS.json) / 2 = TF32 rate"
    else:
        peak, peak_src = 1125.0, "fallback: nominal dense TF32 = 2250 / 2 TFLOP/s (B200_PROFILING.md)"
    ach = S * BLOCK * flop / (fir_ms * 1e-3) / 1e12

    def streaming(D, h):
        # (geometry of the stage's band, served by the streaming kernel?)  Its signature: 64-output tiles and a tap count padded to
        # D + lead chunks, lead <= two tiles' worth of chunks (fir_long_tc.cu: tcs_applies)
        try:
            g, _, _ = engine.long_tc_band(D, h)
        except engine.NvxError:
            return None, False   # the stage runs on CUDA cores
        cs = 32 // D * D
        cpt, lead = D * g["n_tile"] // cs, g["chunks"] - D * g["n_tile"] // cs
        return g, g["n_tile"] == 64 and 0 <= lead <= 2 * cpt and g["taps_padded"] == D + lead * cs

    def executed_tflop(D, h, rows, n_in):
        # what the tensor cores execute for one stage (fir_long_tc.cu geometry, from the library's own band builder): per 128-row
        # tile of n_tile outputs, `chunks` K chunks of 2 planes x 3 TF32 terms x 4 k-steps of M128 x n_tile x K8
        g, is_streaming = streaming(D, h)
        if g is None:
            return 0.0
        tiles = -(-rows // 128) * -(-(n_in // D) // g["n_tile"])
        cs = 32 // D * D
        cpt, lead = D * g["n_tile"] // cs, g["chunks"] - D * g["n_tile"] // cs
        if is_streaming:         # streaming kernel (two or three live tiles): MMAs trimmed to the non-zero columns of the band, N = 16 .. 64
            opc, cols = cs // D, 0
            for c in range(g["chunks"]):
                n_lo, n_hi = max(0, opc * (c - lead)), min(63, opc * c + opc - 1)
                cols += ((n_hi | 15) + 1) - (n_lo & ~15)
        else:                    # tile-at-a-time kernel: the same trimming from its own window geometry (fir_tc_kernel)
            N, Tp, cols = g["n_tile"], g["taps_padded"], 0
            for c in range(g["chunks"]):
                num = cs * c - Tp + 1
                n_lo, n_hi = (0 if num <= 0 else -(-num // D)), min(N - 1, (cs * c + cs - 1) // D)
                cols += ((n_hi | 15) + 1) - (n_lo & ~15) if n_lo <= n_hi else N
        return tiles * cols * 24 * 2.0 * 128 * 8 / 1e12
    ex = executed_tflop(4, taps[0], S, BLOCK) + executed_tflop(7, taps[1], 2 * S, BLOCK // 4)
    # the HBM side of the same three kernels: input once, y1 (63 kHz) and y2 (9 kHz) written and read back once each.  y1 is ONE
    # un-mixed row per stream when stage 2 mixes while it loads (reference offsets + streaming tensor-core stage 2, the default:
    # engine.cu mix_on_load), else one row per channel
    tc_mask = int(os.environ.get("NVX_LONG_TC", "3"))
    mix_on_load = bool(tc_mask & 2) and streaming(7, taps[1])[1] and os.environ.get("NVX_LONG_MIX") != "stage1"
    hbm_bytes = 8.0 + (1 if mix_on_load else 2) * 2 * 8.0 / 4 + 2 * 2 * 8.0 / 28 + 2 * 8.0 / 280
    hbm_peak, hbm_src = measured_peak()
    hbm_ach = S * BLOCK * hbm_bytes / (fir_ms * 1e-3) / 1e9
    return {
        "value": total / (ms * 1e-3) / 1e6, "unit": "Msamples/s", "steps": steps, "warmup": warmup, "ms_per_step": ms / steps,
        "workload": "configs[4]: long-tap FIR stress, %d-tap Kaiser designs in all three stages, 1024 synthetic IQ streams per GPU resident in HBM "
                    "(21.2 GB float2 per step: larger than L2)" % T,
        "taps": [T, T, T], "dtype": "f32 (stages 1-2: 3xTF32 on tcgen05, FP32 accumulate; NVX_LONG_TC=%s)" % os.environ.get("NVX_LONG_TC", "3 (default)"),
        "blocking_note": "tensor-core stages are deterministic for a given blocking and equal across blockings to rounding (1e-5 bar), not bit for bit",
        "engine_note": note or None, "long_tc_fallbacks": int(st.long_tc_fallbacks),
        "realtime_streams": total / (ms * 1e-3) / 252000,
        "roofline": {"bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak, "peak_source": peak_src,
                     "kernel": "nvx::fir_tc_kernel<4,.> + <7,.> + fir_long_kernel<10,2>", "kernel_ms": fir_ms, **span_stats(spans),
                     "note": "achieved = ALGORITHMIC FP32 flops (%.0f per input sample) / time of the three stage kernels; the tensor cores "
                             "execute 3x that for the TF32 split plus the structural zeros of the Toeplitz band" % flop,
                     "executed_tensor_tflops": ex / (fir_ms * 1e-3), "executed_frac": ex / (fir_ms * 1e-3) / peak,
                     "hbm": {"algorithmic_bytes_per_sample": hbm_bytes, "y1_rows_per_stream": 1 if mix_on_load else 2,
                             "achieved": hbm_ach, "peak": hbm_peak, "unit": "GB/s", "frac": hbm_ach / hbm_peak, "peak_source": hbm_src,
                             "note": "the three stage kernels' compulsory HBM traffic (input + y1 and y2 written and read back once) / "
                                     "their time: the bound that matters for short filters, the tensor figure for long ones"}},
        "gpu_launches": int(st.cascade_launches + st.demod_launches + st.aux_launches), "clocks": clocks,
        "check": {"bulletins_in_capture_all_ranks": exp_all, "decoded_exact_all_ranks": ok_all, "messages_total_all_ranks": n_all},
    }


def leg_channels(c, x, expect):
    """SURVEY.md 8f.4: the cost of more channels per capture sharing stage 1.  The default captures through engines with 2 (the
    reference's table NCO), 2, 3 and 4 channels on per-stream offsets (+14 / -14 kHz and two neighbours): kernel time of the one
    pass against the HBM bound of the same bytes; the bulletins on the first two channels are checked as everywhere."""
    import numpy as np
    from navtex_b200 import engine

    S = STREAMS_PER_GPU
    peak, _ = measured_peak()
    offsets, tags = [14000.0, -14000.0, 7000.0, -21000.0], [518, 490, 511, 483]
    out = []
    for n_ch, general in ((2, False), (2, True), (3, True), (4, True)):
        kw = {}
        if general:
            kw = dict(nco_hz=np.tile(np.array(offsets[:n_ch]), (S, 1)), stream_freq_tag=np.tile(np.array(tags[:n_ch]), (S, 1)), n_channels=n_ch)
        eng = engine.Engine(S, BLOCK, device=c.local, first_stream_id=c.rank * S, **kw)
        ms, st, msgs, clocks, spans = timed_pushes(c, eng, x.data_ptr(), BLOCK, 5, 2)
        ok, _ = count_exact(msgs, expect)
        ok_all, = allreduce_sum(c, [ok])
        eng.close()
        k_ms = st.cascade_ms / max(1, st.cascade_launches)
        bytes_alg = S * BLOCK * (8.0 + n_ch * 8.0 / 280)
        out.append({"channels": n_ch, "nco": "per-stream offsets (exact integer phase)" if general else "reference 9-entry table",
                    "kernel_ms": k_ms, **span_stats(spans), "ms_per_step": ms / 5, "value": c.world * S * BLOCK * 5 / (ms * 1e-3) / 1e6,
                    "hbm_frac": bytes_alg / (k_ms * 1e-3) / 1e9 / peak, "decoded_exact_all_ranks": ok_all})
    return {"unit": "Msamples/s", "what": "fused kernel with n channels per capture sharing stage 1, 5 timed steps each, same captures", "runs": out}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workload", default="config2", choices=["config2", "config4", "config5"],
                    help="config2 (default, the metric's configuration, with short config4 / config5 passes folded into the line); "
                         "config4: 8192 streams/GPU x --seconds of traffic generated on the device block by block (BASELINE.json "
                         "configs[3]) as the whole line; config5: the default captures through --taps-tap filters (configs[4])")
    ap.add_argument("--taps", type=int, default=255, help="config5: taps per stage")
    ap.add_argument("--seconds", type=float, default=60.0, help="--workload config4: traffic per stream")
    ap.add_argument("--skip", default="", help="comma-separated legs to leave out of the default line: parity,int16,e2e,config4,config5,channels,cpu")
    ap.add_argument("--parity-streams", type=int, default=PARITY_STREAMS,
                    help="streams of the workload compared against the unmodified reference in the same run (check.oracle_parity); up to 1024")
    ap.add_argument("--pinned", default="nvx", choices=["nvx", "wc"], help="e2e host buffer: cudaHostAlloc portable (nvx) or write-combined (wc)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what their last step computed to DIR/*.npy (rank 0's streams; see dump_outputs)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "b200" or args.workload != "config2"):
        ap.error("--dump-outputs applies to the default workload of --impl b200")
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    skip = set(filter(None, args.skip.split(",")))

    if args.impl == "reference":
        impl_reference(args, rank, world)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    from navtex_b200 import engine, sharding

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (this framework has no CPU path; use --impl reference for the CPU chain)")
    torch.cuda.set_device(local)
    c = Ctx()
    c.torch, c.dist, c.rank, c.world, c.local = torch, dist, rank, world, local
    c.device = torch.device("cuda", local)
    c.cpus = bind_cpus(local, world) if world > 1 else None
    if world > 1:
        # stdout carries exactly one JSON line: NCCL prints its version banner (and anything else NCCL_DEBUG asks for) to
        # stdout unless told otherwise
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=c.device)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    c.barrier = barrier
    c.sampler = ClockSampler(local) if rank == 0 else None

    def finish():
        if c.sampler:
            c.sampler.close()
        if world > 1:
            dist.destroy_process_group()

    base = {"metric": "iq_msamples_per_s", "unit": "Msamples/s", "n_gpus": world, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "data": "synthetic"}

    if args.workload == "config4":
        rec = leg_config4(c, args.seconds, standalone=True)
        if rank == 0:
            print(json.dumps({**base, "value": rec.pop("value"), "steps": rec.pop("steps"), "warmup": 1, "ms_per_step": rec.pop("ms_per_step"),
                              "dtype": "f32", "config": {"workload": rec.pop("workload"), "streams_per_gpu": C4_STREAMS,
                                                         "samples_per_stream_per_step": C4_BLOCK, "parallelism": f"stream-sharded x{world}, no collectives"},
                              **rec, "e2e": None, "cpu_baseline": None}), flush=True)
        finish()
        return

    S = STREAMS_PER_GPU
    x, expect = build_workload(torch, c.device, rank)

    if args.workload == "config5":
        rec = leg_config5(c, x, expect, args.taps, args.steps, args.warmup)
        if rank == 0:
            print(json.dumps({**base, "value": rec.pop("value"), "steps": rec.pop("steps"), "warmup": rec.pop("warmup"), "ms_per_step": rec.pop("ms_per_step"),
                              "dtype": rec.pop("dtype"), "config": {"workload": rec.pop("workload"), "streams_per_gpu": S, "samples_per_stream_per_step": BLOCK,
                                                                    "taps": rec.pop("taps"), "parallelism": f"stream-sharded x{world}, no collectives"},
                              **rec, "e2e": None, "cpu_baseline": None}), flush=True)
        finish()
        return

    # ---- device-resident whole-job throughput ----------------------------------------------------
    eng = engine.Engine(S, BLOCK, device=local, first_stream_id=rank * S)
    max_ms, st, msgs, clocks, spans = timed_pushes(c, eng, x.data_ptr(), BLOCK, args.steps, args.warmup)
    if args.dump_outputs and rank == 0:
        dump_outputs(eng, args.dump_outputs)
    # demod stage breakdown from a short extra pass (the per-stage event records would only add bubbles to the timed region)
    eng.enable_timing(2)
    eng.stats()
    for _ in range(3):
        eng.push_device(x.data_ptr(), BLOCK)
    st2 = eng.stats()
    eng.poll_messages()
    eng.close()
    # correctness of what was timed: each pass over the block re-decodes every stream's bulletin.  EVERY rank checks its own.
    total_samples = world * S * BLOCK * args.steps
    value = total_samples / (max_ms * 1e-3) / 1e6                     # Msamples/s
    decoded_ok, multiset_ok, check = verify_all_ranks(c, msgs, expect, args.steps)

    # ---- same-run parity against the unmodified reference (rank 0's streams) ----------------------
    oracle_parity = None
    if rank == 0 and "parity" not in skip:
        oracle_parity = leg_oracle_parity(c, x, expect, args.parity_streams)
    barrier()

    # ---- secondary: the same captures resident as int16 I,Q (the radio's own format), fused-ingest kernel variant ----
    int16_input, ok16 = None, 0
    if "int16" not in skip:
        x16 = x.round().to(torch.int16)
        eng16 = engine.Engine(S, BLOCK, device=local, first_stream_id=rank * S)
        k16 = min(args.steps, 20)
        t16, st16, msgs16, clocks16, spans16 = timed_pushes(c, eng16, x16.data_ptr(), BLOCK, k16, args.warmup, s16=True)
        ok16, _ = count_exact(msgs16, expect)
        casc16_ms = st16.cascade_ms / max(1, st16.cascade_launches)
        int16_input = {
            "value": world * S * BLOCK * k16 / (t16 * 1e-3) / 1e6, "unit": "Msamples/s", "steps": k16,
            "ms_per_step": t16 / k16, "kernel": "nvx::fir_cascade_kernel<true,false,true,0> (short2 rows by TMA, PRMT/FADD2 conversion)",
            "kernel_ms": casc16_ms, **span_stats(spans16), "algorithmic_bytes_per_sample": 4.0 + 16.0 / 280,
            "achieved_gbs": S * BLOCK * (4.0 + 16.0 / 280) / (casc16_ms * 1e-3) / 1e9, "bound": "fp32 issue (not HBM)",
            # 55.5 algorithmic flop per input sample (SURVEY.md 8d) against 148 SMs x 128 lanes x 2 x 1.965 GHz = 74.5 TFLOP/s
            "fp32_tflops": S * BLOCK * 55.5 / (casc16_ms * 1e-3) / 1e12, "fp32_frac_of_peak": S * BLOCK * 55.5 / (casc16_ms * 1e-3) / 74.5e12,
            "clocks": clocks16,
        }
        eng16.close()
        del x16, eng16

    cpu_sample = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline and "cpu" not in skip:
        n_cpu = 4 * 252000
        cpu_sample = [x[k, :n_cpu].round().to(torch.int16).cpu().numpy().reshape(-1) for k in range(0, S, S // 64)][:64]

    # ---- end to end through the host-buffer C ABI --------------------------------------------------
    e2e, n_e2e, e2e_exact, e2e_expected = None, 0, 0, 0
    if "e2e" not in skip:
        e2e, n_e2e, e2e_exact, e2e_expected = leg_e2e(c, x, expect, args)

    # ---- BASELINE configs[4] and configs[3], short passes in front of the driver ------------------
    channels = leg_channels(c, x, expect) if "channels" not in skip else None
    config5 = leg_config5(c, x, expect, args.taps, 5, 2) if "config5" not in skip else None
    del x
    torch.cuda.empty_cache()
    config4 = leg_config4(c, 10.0) if "config4" not in skip else None

    sums = allreduce_sum(c, [decoded_ok, len(expect), multiset_ok, ok16, n_e2e, e2e_exact, e2e_expected])
    if rank != 0:
        finish()
        return
    check.update({"decoded_exact_all_ranks": sums[0], "bulletins_expected_all_ranks": sums[1], "ranks_with_exact_multiset": sums[2],
                  "int16_decoded_exact_all_ranks": sums[3] if int16_input else None,
                  "e2e_messages_all_ranks": sums[4], "e2e_messages_exact_all_ranks": sums[5], "e2e_bulletins_completed_in_timed_steps_all_ranks": sums[6],
                  "oracle_parity": oracle_parity,
                  "y3_max_rel_err": oracle_parity["y3_max_rel_pair_peak"] if oracle_parity else None})

    # ---- roofline of the dominant kernel (fused FIR cascade) -------------------------------------------
    peak, peak_src = measured_peak()
    casc_ms = st.cascade_ms / max(1, st.cascade_launches)
    achieved = S * BLOCK * BYTES_PER_SAMPLE / (casc_ms * 1e-3) / 1e9
    traffic = ncu_traffic()
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic["dram_bytes_per_launch"] if traffic else None,
                "traffic_source": {k: traffic.get(k) for k in ("source", "command", "commit", "date", "kernel")} if traffic else None,
                "peak_source": peak_src,
                "kernel": "nvx::fir_cascade_kernel<true,false,false,0>", "kernel_ms": casc_ms, **span_stats(spans),
                "whole_step_frac": S * BLOCK * BYTES_PER_SAMPLE / (max_ms / args.steps * 1e-3) / 1e9 / peak,
                "demod_chain_ms": st2.demod_ms / max(1, st2.cascade_launches),
                "demod_stage_ms": dict(zip(("angle_corr", "offset_sum", "(history carry: folded into angle_corr)", "symbol_clock", "bit_decide", "fsm"),
                                           (v / max(1, st2.cascade_launches) for v in st2.demod_stage_ms))),
                "algorithmic_bytes_per_launch": S * BLOCK * BYTES_PER_SAMPLE,
                "kernel_gsamples_per_s": S * BLOCK / (casc_ms * 1e-3) / 1e9}

    # ---- CPU baseline: the reference's own chain on the host cores, bounded sample ------------------
    cpu = None
    if cpu_sample is not None:
        cpu, _ = cpu_reference_figures(cpu_sample, 2, 10)

    line = {
        **base, "value": value, "steps": args.steps, "warmup": args.warmup, "ms_per_step": max_ms / args.steps, "dtype": "f32",
        "config": {"workload": "configs[1]: 1024 synthetic IQ streams per GPU through fused FIR cascade + FSK demod + bit-sync + SITOR-B",
                   "streams_per_gpu": S, "samples_per_stream_per_step": BLOCK, "seconds_per_step": BLOCK / 252000,
                   "input": "float2 IQ resident in HBM, 21.2 GB per GPU per step (larger than L2; no flush needed)",
                   "parallelism": f"stream-sharded x{world}, no collectives"},
        "realtime_streams": value / 0.252,
        "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "int16_input": int16_input, "config4": config4, "config5": config5, "channels": channels,
        "gpu_launches": int(st.cascade_launches + st.demod_launches + st.aux_launches),
        "clocks": clocks,
        "check": check,
    }
    print(json.dumps(line), flush=True)
    finish()


if __name__ == "__main__":
    main()

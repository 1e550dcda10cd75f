"""The demodulator kernels (demod.cu: angle_corr, offset_sum, symbol_clock, bit_decide, fsm) bit for bit against the oracle fed
at 900 Hz (oracle_lib.run_oracle_900).

An engine with unit taps, one channel and a 0 Hz NCO passes each 900 Hz sample, repeated over its 280 input samples, through
the cascade unchanged (checked at every block), so the demodulator sees exactly the rows of demod_inputs.py.  Only FP64 atan2
may differ between the GPU and the host C library (within 2 ulp).  So:
  lattice rows (every angle an exact special value of atan2): bits, discriminator sums (bitwise), events and messages equal;
  other rows: equal too, except from the first decision that follows an oracle arg max pick margin below 1e-12 within the 64
  evaluations before it (attributed as tests/parity.py does, and recorded in the parity report).
S = 1057 rows: three CTAs of the lane-per-channel kernels, a last warp with one live lane, a ragged offset_sum unit count.
Block lengths (in 900 Hz samples) run from 1 to 4700, end on every residue mod 9 and mod 567 and at 573 .. 583 (the ring fills,
the first evaluation falls), and cross the 256-evaluation / 256-bit chunks of the sequential kernels inside a block and at its
end.  Rows are reset mid-run (one warp then mixes epochs), and a ragged set is saved and loaded into a second engine."""
import concurrent.futures as cf

import numpy as np
import pytest

import demod_inputs as di
import parity
from navtex_b200 import engine

pytestmark = pytest.mark.gpu

S = 1057
SEED = 2024
BLK = engine.BLOCK_ALIGN
RING = 567                                  # the reset grid at 900 Hz (158 760 input samples)
MAX_N = 4700
NEAR_TIE = 1e-12


def schedule():
    """(block lengths, index of the save, {block index: rows reset before it})"""
    rng = np.random.default_rng(SEED)
    b = [1, 2, 7, 8, 9, 10, 63, 255, 218] + [1] * 10            # ends 1 .. 573, then 574 .. 583
    b += [256, 257, 566, 567, 568, 2303, 2304, 2305, 4700]
    resets = {len(b): [3, 40, 511, 512, 1056]}
    b += [3001]
    b += list(rng.integers(1, 2 * RING, 24))
    resets[len(b)] = [4, 41, 100, 1055, 600]
    b += [4700, 2600]
    save = len(b)
    b += [1] * 300                                              # a run of single-sample blocks
    b += list(rng.integers(1, MAX_N + 1, 6))
    ends = set(np.cumsum(b) % RING)
    while len(ends) < RING:                                     # then land on every residue mod 567 not yet hit
        end = int(np.sum(b))
        n = min((r - end) % RING or RING for r in range(RING) if r not in ends)
        b.append(n + RING * int(rng.integers(0, 2)))
        ends.add((end + b[-1]) % RING)
    return [int(n) for n in b], save, resets


def test_schedule_reaches_the_edges():
    b, save, resets = schedule()
    ends = np.cumsum(b)
    assert set(ends % 9) == set(range(9)) and set(ends % RING) == set(range(RING))
    assert set(range(573, 584)) <= set(ends.tolist())
    assert {255, 256, 257, 2303, 2304, 2305, 4700} <= set(b) and max(b) <= MAX_N
    assert all(b[k] > 2304 for k in resets)


def _oracle_rows(rows_x):
    import oracle_lib as ol
    ol.lib()
    with cf.ThreadPoolExecutor() as ex:
        return list(ex.map(ol.run_oracle_900, rows_x))


class _Run:
    """per row: the GPU's bits, discriminator sums and events, block by block"""

    def __init__(self, eng, rows):
        self.eng, self.rows = eng, rows
        self.bits = {r: [] for r in rows}
        self.disc = {r: [] for r in rows}
        self.ev = {r: [] for r in rows}
        self.msgs = []

    def push(self, X, x_host, pos, n):
        import torch
        dev = torch.repeat_interleave(X[:, pos:pos + n], BLK, dim=1).contiguous()     # [S, 280 n, 2] float32
        torch.cuda.synchronize()
        self.eng.push_device(dev.data_ptr(), n * BLK)
        assert self.eng.L.nvx_engine_sync(self.eng._h) == 0, engine.load_library().nvx_last_error()     # no overflow
        del dev
        y3 = self.eng.read_y3()[:, 0]
        assert np.array_equal(y3.view(np.uint64), x_host[:, pos:pos + n].view(np.uint64)), ("y3 is not the input", pos, n)
        for r in self.rows:
            bits, sums = self.eng.read_bits(r, 0)
            self.bits[r].append(bits)
            self.disc[r].append(sums)
            self.ev[r].append(self.eng.read_events(r, 0))
        self.msgs += self.eng.poll_messages(wait=False)

    def row(self, r, first_block=0, last_block=None):
        sl = slice(first_block, last_block)
        d = self.disc[r][sl]
        return (b"".join(self.bits[r][sl]), np.concatenate(d) if d else np.zeros((0, 4), np.float32), b"".join(self.ev[r][sl]))


def _check(where, got, ref, lattice, stats):
    """got: (bits, disc, events, messages [(bbbb, text)]); ref: an oracle Result.  Returns True when compared in full."""
    bits, disc, ev, msgs = got
    t = "518"
    rb, rd = ref.bits[t], ref.disc[t]
    m = min(len(bits), len(rb))
    diff = np.frombuffer(bits[:m], np.uint8) != np.frombuffer(rb[:m], np.uint8)
    diff |= (disc[:m].view(np.uint32) != rd[:m].view(np.uint32)).any(axis=1)
    if len(bits) != len(rb):
        diff = np.append(diff, True)
    pm = ref.pick_margins[t]
    if not diff.any():
        assert ev == ref.events[t], (where, "events", ev[-40:], ref.events[t][-40:])
        assert msgs == ref.messages, (where, "messages", msgs, ref.messages)
        return True
    k = int(np.argmax(diff))
    assert not lattice, (where, "lattice row differs at decision", k, len(bits), len(rb))
    at = np.searchsorted(pm[:, 0], ref.bitpos[t][min(k, len(rb) - 1)], side="right") if len(rb) else 0
    tight = float(pm[max(0, at - 64):at, 1].min()) if at else np.inf
    assert tight < NEAR_TIE, (where, "decision", k, "differs; tightest pick margin before it", tight)
    cmp = parity.compare_stream([ref.y3[t]], [bits], [disc], ref, occupied=(), channels=(t,))
    parity.record(where, cmp, occupied=())
    stats["excusals"].append((where, k, tight))
    return False


def test_demodulator_kernels_bit_for_bit(oracle):
    import torch
    blocks, save, resets = schedule()
    N = sum(blocks)
    rows = [di.row(SEED, r, N) for r in range(S)]
    x_host = np.stack([x for x, _ in rows])
    meta = [m for _, m in rows]
    X = torch.from_numpy(x_host.view(np.float32).reshape(S, N, 2)).cuda()
    starts = np.concatenate([[0], np.cumsum(blocks)])

    mk = lambda: engine.Engine(S, MAX_N * BLK, keep_bits=True, taps=([1.0], [1.0], [1.0]), nco_hz=np.zeros((S, 1)),
                               stream_freq_tag=np.full((S, 1), 518), n_channels=1)
    rng = np.random.default_rng(SEED + 1)
    reset_rows = {r: k for k, rs in resets.items() for r in rs}
    saved = sorted({int(r) for r in rng.choice(S, 300, replace=False)} | set(range(640, 700)))
    saved = [r for r in saved if r not in reset_rows]
    a, b = _Run(mk(), range(S)), None
    for i, n in enumerate(blocks):
        if i in resets:
            a.eng.reset_streams(resets[i])
        if i == save:
            state = a.eng.save_streams(saved)
            b = _Run(mk(), range(S))
            b.eng.load_streams(saved, state)
        a.push(X, x_host, int(starts[i]), n)
        if b is not None:
            b.push(X, x_host, int(starts[i]), n)
    a.msgs += a.eng.poll_messages()
    b.msgs += b.eng.poll_messages()
    a.eng.close()
    b.eng.close()

    # the oracle runs: uninterrupted rows; rows restarted at E (a fresh decoder fed E mod 567 zeros, then the row from E on); and
    # the prefixes before E, which split an uninterrupted row's events and messages at E
    e_save = int(starts[save])
    jobs = {("full", r): x_host[r] for r in range(S)}
    for r, k in reset_rows.items():
        e = int(starts[k])
        jobs[("fresh", r)] = np.concatenate([np.zeros(e % RING, np.complex64), x_host[r, e:]])
        jobs[("pre", r)] = x_host[r, :e]
    for r in range(S):
        if r in saved:
            jobs[("pre_save", r)] = x_host[r, :e_save]
        else:
            jobs[("fresh_save", r)] = np.concatenate([np.zeros(e_save % RING, np.complex64), x_host[r, e_save:]])
    keys = list(jobs)
    ref = dict(zip(keys, _oracle_rows([jobs[k] for k in keys])))

    stats = {"ties": 0, "min_margin": np.inf, "excusals": []}
    msgs_of = lambda run, r: [(f, bb, tx) for s, f, bb, tx in run.msgs if s == r]
    full = 0
    for r in range(S):
        lat = meta[r]["family"] == "lattice"
        pm = ref[("full", r)].pick_margins["518"][:, 1]
        stats["ties"] += int((pm == 0).sum())
        if not lat:         # exact zeros come from silence (all nine sums 0), where both sides agree; the smallest non-zero margin is
            stats["min_margin"] = min(stats["min_margin"], float(pm[pm > 0].min(initial=np.inf)))     # what a flip needs
        if r in reset_rows:
            k = reset_rows[r]
            pre, fresh = ref[("pre", r)], ref[("fresh", r)]
            bits, disc, ev = a.row(r, 0, k)
            mine = msgs_of(a, r)
            npre = len(pre.messages)
            _check(("A", r, "before reset"), (bits, disc, ev, mine[:npre]), pre, lat, stats)
            full += _check(("A", r, "after reset"), a.row(r, k) + (mine[npre:],), fresh, lat, stats)
        else:
            full += _check(("A", r), a.row(r) + (msgs_of(a, r),), ref[("full", r)], lat, stats)
        if r in saved:      # B continues the uninterrupted row: its decisions after E, its events and messages after the prefix's
            o, p = ref[("full", r)], ref[("pre_save", r)]
            bits, disc, ev = b.row(r)
            got = (p.bits["518"] + bits, np.concatenate([p.disc["518"], disc]), p.events["518"] + ev,
                   p.messages + msgs_of(b, r))
            _check(("B", r, "loaded"), got, o, lat, stats)
        else:
            _check(("B", r, "restarted at the load"), b.row(r) + (msgs_of(b, r),), ref[("fresh_save", r)], lat, stats)

    # coverage: the inputs still reach the edges
    ev_all = [a.row(r)[2] for r in range(S)]
    gaps = set()
    for r in range(S):
        if meta[r]["family"] == "fsk":
            gaps |= set(np.diff(ref[("full", r)].bitpos["518"]).tolist())
    parity.REPORT.append({"where": "test_gpu_demod", "rows": S, "blocks": len(blocks), "samples_900hz": N, "exact_ties": stats["ties"],
                          "near_tie_excusals": stats["excusals"], "min_nonzero_pick_margin_non_lattice": stats["min_margin"],
                          "rows_compared_in_full": full})
    assert stats["ties"] >= 1000, stats["ties"]
    assert {8, 10} <= gaps, gaps
    assert sum(e.count(b"*\x18") for e in ev_all) >= 10
    assert sum(di.eoe_aborts(e) for e in ev_all) >= 100
    assert sum(e.count(b"*") for e in ev_all) >= 100
    assert len(a.msgs) >= 150, len(a.msgs)

#!/usr/bin/env python3
"""Generate tests/golden/*.npz by running the UNMODIFIED reference (oracle/_ref/ref_chain, built
from /root/reference by oracle/Makefile) on the deterministic captures of tests/cases.py.

Run in the build container only:   python tests/golden/make_golden.py
The fixtures pin the CPU restatement (oracle/navtex_oracle.c) and the CUDA path on machines where
/root/reference does not exist.  Each fixture stores the SHA-256 of its input capture so a test can
tell "numpy regenerated a different capture" apart from "results differ".
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
Y3_MAX = 24000      # 900 Hz samples of y3 kept per channel (26.7 s): keeps every fixture under 1 MB
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

import cases  # noqa: E402
import oracle_lib  # noqa: E402
from navtex_b200 import synth  # noqa: E402


def main():
    assert oracle_lib.have_ref(), "build oracle/_ref first (make -C oracle ref)"
    for name in cases.CASES:
        iq = cases.build(name)
        r = oracle_lib.run_ref(iq)
        out = dict(sha256=cases.digest(iq), n=iq.size // 2, y1_head=r.y1[:4096])
        for tag in oracle_lib.CHANNELS:
            out["y2_head_" + tag] = r.y2[tag][:2048]
            out["y3_" + tag] = r.y3[tag][:Y3_MAX]
            out["bits_" + tag] = np.frombuffer(r.bits[tag], dtype=np.uint8)
            out["bitpos_" + tag] = r.bitpos[tag]
            out["disc_" + tag] = r.disc[tag]
        out["msg_freq"] = np.array([m[0] for m in r.messages], dtype=np.int32)
        out["msg_bbbb"] = np.array([m[1] for m in r.messages], dtype="U8")
        out["msg_text"] = np.array([m[2] for m in r.messages], dtype="U5000") if r.messages else np.array([], dtype="U1")
        np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
        print(name, out["n"], [len(r.bits[t]) for t in oracle_lib.CHANNELS], r.messages)
    # the WAV input path (wav.c reader) must give the same results as the raw path
    iq = cases.build("clean518")
    wav = "/tmp/navtex_clean518.wav"
    synth.write_wav(wav, iq)
    rw = oracle_lib.run_ref(wav=wav)
    rr = oracle_lib.run_ref(iq)
    assert rw.messages == rr.messages and rw.bits == rr.bits
    for tag in oracle_lib.CHANNELS:
        assert np.array_equal(rw.y3[tag], rr.y3[tag])
    print("wav path == raw path")


if __name__ == "__main__":
    main()

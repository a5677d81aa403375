"""CPU sweep of the frame-synchronous ENCODER PIPELINE's stage functions (celt_enc_pipe.cuh / celt_enc_bandpipe.cuh) through the host
simulation (1-lane teams, the kernels' stage order emulated, tests/hostsim) against the oracle: the full grid of
tests/test_cpu.py::test_hostsim_encoder_pipeline_vs_oracle_mini_sweep (signal x channels x frame size x bitrate x CBR/VBR/CVBR x
complexity = 2,304 cases) instead of its sample of 150, band stage as the inline walk the GPU runs.  A test tool: it checks the integer
logic of the shared headers, not warp-level behaviour.

usage: python tools/hostsim_pipe_sweep.py [workers=8] [seconds_per_stream=0.5]"""
import os
import sys
import time
from multiprocessing import Pool

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import oracle_lib as O

CASES = [(k, ch, fs, br, m, cx) for k in ("music", "tone", "clicks", "noise") for ch in (1, 2) for fs in (120, 240, 480, 960)
         for br in (32000, 48000, 64000, 96000, 128000, 192000, 256000, 510000) for m in ((0, 0), (1, 0), (1, 1)) for cx in (0, 5, 10)]
SECONDS = float(sys.argv[2]) if len(sys.argv) > 2 else 0.5
_hs = None


def run(i):
    global _hs
    import test_cpu as T
    if _hs is None:
        _hs = T._hostsim()
        _hs.hostsim_set_band_mode(2)
    kind, ch, fs, br, (vbr, cvbr), cx = CASES[i]
    x = O.test_signal(int(48000 * SECONDS), ch, 9000 + i, kind)
    d, o, l, r = O.encode_stream(x, fs, br, ch, vbr=vbr, cvbr=cvbr, complexity=cx, max_bytes=1276, pin=False)
    rc, out, lens, rng = T._hostsim_encode_pipe(_hs, x, fs, br, ch, vbr, cvbr, cx, Fc=(1, 2, 3, 8, 16)[i % 5])
    ok = rc == 0 and T._same_packets(d, o, l, out, lens) and np.array_equal(r, rng)
    return i, bool(ok)


if __name__ == "__main__":
    workers = int(sys.argv[1]) if len(sys.argv) > 1 else 8
    t0 = time.time()
    with Pool(workers) as p:
        res = p.map(run, range(len(CASES)), chunksize=16)
    bad = [CASES[i] for i, ok in res if not ok]
    print("hostsim pipeline sweep: %d cases x %.1f s, inline walk: %d mismatching, %.0f s" % (len(CASES), SECONDS, len(bad), time.time() - t0))
    for b in bad[:20]:
        print("  BAD", b)
    sys.exit(1 if bad else 0)

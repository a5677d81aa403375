"""Randomised encoder ctl sweep on the GPU: every stream of a batch follows its own random script of opus_encoder_ctl changes
(bitrate, VBR, CVBR, complexity, forced channels, bandwidth / max bandwidth, packet-loss %, LSB depth, prediction-disabled,
forced mode, OPUS_RESET_STATE: the reference's own fuzz shape, opus-fix/tests/test_opus_encode.c:236-330) while the whole batch is
coded through opus_encode_span one frame per call — so states hop between HBM residency (span) and the host (ctl) all the time.
Packets, lengths and final range after every frame vs the oracle run with the same script.

usage: python tools/parity_sweep_ctl.py [batches=12] [streams=32] [seed=1]
"""
import ctypes as C
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import concentus_b200 as cb
import oracle_lib as O

NB = int(sys.argv[1]) if len(sys.argv) > 1 else 12
NS = int(sys.argv[2]) if len(sys.argv) > 2 else 32
SEED = int(sys.argv[3]) if len(sys.argv) > 3 else 1
L = cb.lib()
assert L.opus_b200_init(0) == 0
rs = np.random.RandomState(SEED)
KINDS = ("music", "tone", "clicks", "noise")
bad_total, t0 = 0, time.time()
for b in range(NB):
    ch = int(rs.choice([1, 2]))
    fs = int(rs.choice([120, 240, 480, 960]))
    F = 60
    seeds = [int(rs.randint(1 << 30)) for _ in range(NS)]
    pcms = [O.test_signal(F * fs, ch, sd, KINDS[sd % 4]) for sd in seeds]
    scripts = [O.ctl_script(sd, F, ch, K=2) for sd in seeds]
    refs = [O.encode_stream_script(pcms[i], fs, ch, scripts[i], pin=False) for i in range(NS)]
    enc = cb.EncoderBatch(NS, 48000, ch, bitrate=64000, vbr=1, cvbr=1, complexity=10)
    x = np.stack([p.reshape(F, fs * ch) for p in pcms])
    v = C.c_uint32(0)
    bad = set()
    for f in range(F):
        for i in range(NS):
            hp = C.c_void_p(enc.handles[i])
            for (req, val) in scripts[i][f]:
                if req == 4028:
                    L.opus_encoder_ctl(hp, 4028)
                elif req:
                    L.opus_encoder_ctl(hp, int(req), C.c_int32(int(val)))
        d, l = enc.encode_span(np.ascontiguousarray(x[:, f]).reshape(-1, ch), 1, fs)
        d = d.reshape(NS, 1276)
        for i in range(NS):
            rd, rl, rr = refs[i]
            n = int(l[i])
            if n != int(rl[f]) or not np.array_equal(d[i, :max(n, 0)], rd[f, :max(n, 0)]):
                bad.add(i)
        if f % 7 == 3:   # final range through a ctl (pulls the state back to the host) for a few streams
            for i in range(0, NS, 5):
                L.opus_encoder_ctl(C.c_void_p(enc.handles[i]), cb.OPUS_GET_FINAL_RANGE_REQUEST, C.byref(v))
                if v.value != int(refs[i][2][f]):
                    bad.add(i)
    enc.close()
    bad_total += len(bad)
    print("batch %2d: ch=%d frame=%4d  streams with a mismatch: %d %s" % (b, ch, fs, len(bad), sorted(bad)[:6]), flush=True)
print("ctl sweep: %d batches x %d streams x 60 frames, seed %d: %d mismatching streams, %.0f s" % (NB, NS, SEED, bad_total, time.time() - t0))
sys.exit(1 if bad_total else 0)

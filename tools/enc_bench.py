"""Dev tool: encoder throughput on the GPU (kernel time from CUDA events inside the library)."""
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import concentus_b200 as cb
import oracle_lib as O

n = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
F = int(sys.argv[2]) if len(sys.argv) > 2 else 50
br = int(sys.argv[3]) if len(sys.argv) > 3 else 96000
fs, ch = 960, 2
L = cb.lib()
assert L.opus_b200_init(0) == 0
if os.environ.get("ENC_PATH") == "one_kernel":
    L.opus_b200_enc_set_pipeline(0)
uniq = min(n, 64)
base = [O.test_signal(fs * F, ch, 500 + i, ("music", "tone", "clicks", "music")[i % 4]) for i in range(uniq)]
pcm = np.concatenate([base[i % uniq] for i in range(n)])
enc = cb.EncoderBatch(n, 48000, ch, bitrate=br, vbr=1, cvbr=0, complexity=10)
best = 1e30
for rep in range(int(os.environ.get("REPS", "3"))):
    t0 = time.time()
    d, l = enc.encode_span(pcm, F, fs)
    t1 = time.time()
    ms = L.opus_b200_enc_last_kernel_ms()
    audio_s = n * F * fs / 48000.0
    print("rep %d: kernel %.1f ms -> %.0fx realtime (e2e %.0fx), mean packet %.1f B, errors %d" % (
        rep, ms, audio_s / (ms * 1e-3), audio_s / (t1 - t0), l[l > 0].mean(), int((l < 0).sum())))
    if rep > 0: best = min(best, ms)
print("best kernel %.1f ms -> %.0fx realtime" % (best, audio_s / (best * 1e-3)))
# spot-check parity on a few streams (first span only is comparable: the state carried on)
enc.close()
enc = cb.EncoderBatch(n, 48000, ch, bitrate=br, vbr=1, cvbr=0, complexity=10)
d, l = enc.encode_span(pcm, F, fs)
enc.close()
d = d.reshape(n, F, -1)
l = l.reshape(n, F)
bad = 0
for s in list(range(0, n, max(1, n // 16)))[:16]:
    rd, ro, rl, _ = O.encode_stream(base[s % uniq], fs, br, ch, vbr=1, cvbr=0, complexity=10, pin=False)
    rd = rd.reshape(F, 1276)
    ok = np.array_equal(rl, l[s]) and all(np.array_equal(rd[f, :rl[f]], d[s, f, :rl[f]]) for f in range(F))
    bad += not ok
print("parity spot-check: %d bad of 16" % bad)
import ctypes as C
m, lv = C.c_longlong(0), C.c_longlong(0)
try:
    L.opus_b200_enc_band_stats(C.byref(m), C.byref(lv))
    print("split band loop: %d leaves listed, %d searched by the exact chain (%.2f %%)" % (lv.value, m.value, 100.0 * m.value / max(1, lv.value)))
except Exception as ex:
    print("no band stats:", ex)

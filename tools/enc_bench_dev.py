"""Dev tool: encoder throughput with PCM and packets resident in HBM (opus_encode_span_device), CUDA events on the library's stream.

usage: python tools/enc_bench_dev.py [streams] [frames] [bitrate]      REPS=n for more timed repetitions
The signal mix is tools/enc_bench.py's (music / tone / clicks), `skip` frames into each signal so that the timed span is busy audio."""
import ctypes as C
import os
import sys

import numpy as np
import torch

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
dev = torch.device("cuda:0")
uniq = min(n, 64)
base = [O.test_signal(fs * F, ch, 500 + i, ("music", "tone", "clicks", "music")[i % 4]) for i in range(uniq)]
pcm = np.stack([base[i % uniq] for i in range(n)])
d_pcm = torch.from_numpy(pcm).to(dev).contiguous()
stride = 1276
d_data = torch.zeros((n * F * stride,), dtype=torch.uint8, device=dev)
d_ret = torch.zeros((n * F,), dtype=torch.int32, device=dev)
estream = torch.cuda.ExternalStream(L.opus_b200_enc_stream(), device=dev)
best = 1e30
for rep in range(int(os.environ.get("REPS", "4"))):
    enc = cb.EncoderBatch(n, 48000, ch, bitrate=br, vbr=1, cvbr=0, complexity=10)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record(estream)
    rc = L.opus_encode_span_device(enc.handles, n, F, C.c_void_p(d_pcm.data_ptr()), fs, C.c_void_p(d_data.data_ptr()), stride, C.c_void_p(d_ret.data_ptr()))
    e1.record(estream)
    torch.cuda.synchronize()
    assert rc == 0, rc
    ms = e0.elapsed_time(e1)
    if rep > 0:
        best = min(best, ms)
    if rep == 0:   # parity spot check of the first launch against the oracle
        data = d_data.cpu().numpy().reshape(n, F, stride)
        lens = d_ret.cpu().numpy().reshape(n, F)
        bad = 0
        for s in list(range(0, n, max(1, n // 16)))[:16]:
            rd, ro, rl, _ = O.encode_stream(base[s % uniq], fs, br, ch, vbr=1, cvbr=0, complexity=10, pin=False)
            rd = rd.reshape(F, 1276)
            ok = np.array_equal(rl, lens[s]) and all(np.array_equal(rd[f, :rl[f]], data[s, f, :rl[f]]) for f in range(F))
            bad += not ok
    enc.close()
audio_s = n * F * fs / 48000.0
print("best %.2f ms = %.1f us/frame -> %.0fx realtime, parity %d bad of 16, errors %d" % (best, 1e3 * best / F, audio_s / (best * 1e-3), bad, int((d_ret < 0).sum().item())))

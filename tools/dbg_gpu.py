import sys, os, numpy as np
sys.path.insert(0, os.path.join(os.path.dirname(__file__), '..')); sys.path.insert(0, os.path.join(os.path.dirname(__file__), '..', 'tests'))
import concentus_b200 as cb, oracle_lib as O
L = cb.lib(); assert L.opus_b200_init(0) == 0
n, fs = 2, 960
datas, offs, lens = [], [], []; base = 0
for s in range(n):
    pcm = O.test_signal(48000 // 2, 2, 1000 + s, "music")
    d, o, l, _ = O.encode_stream(pcm, fs, 64000); d, o = O.pack(d, o, l)
    datas.append(d); offs.append(o + base); lens.append(l); base += len(d)
data, offs, lens = np.concatenate(datas), np.concatenate(offs), np.concatenate(lens)
F = len(lens) // n
dec = cb.DecoderBatch(n, 48000, 2)
pcm, rets = dec.decode_span(data, offs, lens, F, fs)
print("rets", rets.reshape(n, F))
for s in range(n):
    sl = slice(s * F, (s + 1) * F)
    rp, rr, _ = O.decode_stream(data, offs[sl], lens[sl], fs, 2, pin=False)
    mine = pcm[s * F * fs:(s + 1) * F * fs]
    bad = np.nonzero((rp.reshape(F, -1) != mine.reshape(F, -1)).any(axis=1))[0]
    print("stream", s, "bad frames", bad)

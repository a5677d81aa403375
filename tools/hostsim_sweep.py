"""CPU twin of tools/parity_sweep.py: the same random batches (draw_batch, wide mode), coded by the HOST SIMULATION of the kernel
headers (tests/hostsim: 1-lane teams, the kernels' call / run schedule emulated) instead of the GPU, against the oracle.  A test
tool like the host simulation itself: it localises logic errors of the shared headers without GPU time; it says nothing about
warp-level races.  Random batches have no stored reference results (tests/oracle_lib.py): run standalone, the oracle is the host
simulation itself, so the sweep checks the emulated call / run schedule against plain per-packet decoding, not the headers' logic.

usage: python tools/hostsim_sweep.py [batches=20] [streams_per_batch=16] [seed=1] [workers=8]
"""
import ctypes as C
import functools
import os
import sys
import time
from multiprocessing import Pool

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import oracle_lib as O
import parity_sweep as PS

_hs = None


def hostsim():
    global _hs
    if _hs is None:
        import test_cpu as T
        _hs = T._hostsim()
        _hs.hostsim_decode_stream_calls.argtypes = [C.c_void_p] * 3 + [C.c_int] * 4 + [C.c_void_p] * 3 + [C.c_void_p, C.c_int]
    return _hs


def one_stream(job, pin=True):
    (b, i, ch, fs, F, cfg, cut, loss, Fs, dFs, dch, maxb, extra, capmul) = job
    hs = hostsim()
    br, (vbr, cvbr), cx, kind, sd = cfg
    pcm = O.test_signal(F * fs, ch, sd, kind)
    rd, ro, rl, rr = PS.ref_encode(pcm, fs, br, ch, Fs, vbr, cvbr, cx, maxb, extra[0], extra[1], pin=pin)
    out = np.zeros((F, 1276), dtype=np.uint8)
    lens = np.zeros(F, dtype=np.int32)
    rng = np.zeros(F, dtype=np.uint32)
    c = np.array([O.OPUS_APPLICATION_RESTRICTED_LOWDELAY, br, vbr, cvbr, cx, maxb, extra[0], extra[1]], dtype=np.int32)
    hs.hostsim_encode_stream(O.ptr(np.ascontiguousarray(pcm)), F, fs, ch, Fs, O.ptr(c), O.ptr(out), 1276, O.ptr(lens), O.ptr(rng))
    rd2 = rd.reshape(F, 1276)
    enc_ok = np.array_equal(rl, lens) and all(np.array_equal(rd2[f, :max(rl[f], 0)], out[f, :max(rl[f], 0)]) for f in range(F)) and \
        int(rr[-1]) == int(rng[-1])
    dl = rl.copy()
    dl[loss == 1] = 0
    dl[loss == 2] = 1
    dfs = int(fs * dFs // Fs * capmul)
    if dfs * 25 > dFs * 3:
        dfs = fs * dFs // Fs
    rp, rrg, rret = O.decode_stream(rd, ro, dl, dfs, dch, Fs=dFs, pin=pin)
    hp = np.zeros((F * dfs, dch), dtype=np.int16)
    hr = np.zeros(F, dtype=np.uint32)
    hret = np.zeros(F, dtype=np.int32)
    bnd = np.array([cut, F], dtype=np.int32)
    hs.hostsim_decode_stream_calls(O.ptr(rd), O.ptr(np.ascontiguousarray(ro, dtype=np.int64)), O.ptr(np.ascontiguousarray(dl, dtype=np.int32)),
                                   F, dfs, dch, dFs, O.ptr(hp), O.ptr(hr), O.ptr(hret), O.ptr(bnd), 2)
    rp = rp.reshape(F, -1)
    hp = hp.reshape(F, -1)
    head_ok = all(np.array_equal(rp[f, :max(int(rret[f]), 0) * dch], hp[f, :max(int(rret[f]), 0) * dch]) for f in range(F))
    dec_ok = np.array_equal(rret, hret) and head_ok and np.array_equal(rrg, hr)
    return (b, i, enc_ok, dec_ok, (ch, fs, Fs, dFs, dch, maxb, capmul, cfg))


def main():
    NB = int(sys.argv[1]) if len(sys.argv) > 1 else 20
    NS = int(sys.argv[2]) if len(sys.argv) > 2 else 16
    SEED = int(sys.argv[3]) if len(sys.argv) > 3 else 1
    NW = int(sys.argv[4]) if len(sys.argv) > 4 else 8
    hostsim()
    rs = np.random.RandomState(SEED)
    jobs = []
    for b in range(NB):
        ch, fs, F, cfgs, cut, loss, Fs, dFs, dch, maxb, extra, capmul = PS.draw_batch(rs, NS, True)
        for i in range(NS):
            jobs.append((b, i, ch, fs, F, cfgs[i], cut, loss[i], Fs, dFs, dch, maxb, extra[i], capmul))
    t0 = time.time()
    bad = 0
    with Pool(NW) as pool:
        for k, (b, i, e_ok, d_ok, info) in enumerate(pool.imap_unordered(functools.partial(one_stream, pin=False), jobs, chunksize=4)):
            if not (e_ok and d_ok):
                bad += 1
                print("MISMATCH batch %d stream %d encode_ok=%s decode_ok=%s %s" % (b, i, e_ok, d_ok, info), flush=True)
            if (k + 1) % 200 == 0:
                print("%d / %d streams, %d mismatching, %.0f s" % (k + 1, len(jobs), bad, time.time() - t0), flush=True)
    print("hostsim sweep: %d batches x %d streams, seed %d: %d mismatching streams, %.0f s" % (NB, NS, SEED, bad, time.time() - t0))
    sys.exit(1 if bad else 0)


if __name__ == "__main__":
    main()

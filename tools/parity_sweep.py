"""Randomised parity sweep on the GPU (beyond the fixed grid of tests/): batches of streams with per-stream random bitrate,
CBR/VBR/CVBR, complexity and signal, for random (channels, frame size); the CUDA encoder against the oracle byte-for-byte, then
the CUDA decoder on the oracle's packets with a random loss pattern against the oracle sample-for-sample.  Prints one line per
batch and a summary; exit code 1 on any mismatch.

usage: python tools/parity_sweep.py [batches=24] [streams_per_batch=48] [seed=1] [wide]     (SWEEP_ONLY=51,123 runs just those batches)
`wide` also draws the encoder's API rate (8-48 kHz), 40 / 60 ms frames (repacketized multi-frame packets), and a decoder whose
rate and channel count differ from the stream's.
Random batches have no stored reference results (tests/oracle_lib.py), so the oracle here is the host simulation of the same
headers unchecked: the sweep finds disagreements between the CUDA and host builds, not errors both share.
"""
import ctypes as C
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
if os.environ.get("SWEEP_PKG"):
    sys.path.insert(0, os.environ["SWEEP_PKG"])   # A/B against an older package + library
import oracle_lib as O

DURATION_MULT = int(os.environ.get("SWEEP_DURATION_MULT", "1"))   # streams of 1-2 s by default; x N for long-horizon state
RATES = [24000, 32000, 40000, 48000, 64000, 80000, 96000, 128000, 160000, 192000, 256000, 320000, 510000]
KINDS = ("music", "tone", "clicks", "noise")


def draw_batch(rs, NS, wide=False):
    """All random parameters of one batch, drawn before any work, so that a batch can be reproduced alone."""
    ch = int(rs.choice([1, 2]))
    fs = int(rs.choice([120, 240, 480, 960]))
    nsec = 2 if fs >= 480 else 1
    F = 48000 * nsec * DURATION_MULT // fs
    if wide:
        Fs = int(rs.choice([8000, 12000, 16000, 24000, 48000]))
        ms10 = int(rs.choice([25, 50, 100, 200, 400, 600]))            # frame duration in 0.1 ms
        fs = Fs * ms10 // 10000
        F = int(Fs * (2 if ms10 >= 100 else 1)) * DURATION_MULT // fs
        dFs = int(rs.choice([8000, 12000, 16000, 24000, 48000]))
        dch = int(rs.choice([1, 2]))
        maxb = int(rs.choice([1276, 1276, 500, 200, 40, 8, 3]))         # max_data_bytes of the batch
        capmul = float(rs.choice([1, 1, 1, 2, 3, 0.5]))                 # decoder PCM capacity per packet / packet duration
        extra = [(int(rs.choice([0, 0, 1, 2])) if ch == 2 else 0,       # OPUS_SET_FORCE_CHANNELS (0 = auto)
                  int(rs.choice([0, 0, 0, 1101, 1102, 1103, 1104, 1105])))   # OPUS_SET_BANDWIDTH (0 = auto)
                 for _ in range(NS)]
    else:
        Fs, dFs, dch, maxb, extra, capmul = 48000, 48000, ch, 1276, [(0, 0)] * NS, 1
    cfgs = [(int(rs.choice(RATES)), [(0, 0), (1, 0), (1, 1)][rs.randint(3)], int(rs.randint(11)), KINDS[rs.randint(4)], int(rs.randint(1 << 30)))
            for _ in range(NS)]
    cut = int(rs.randint(1, F))                       # two spans: state crosses a launch boundary at a random frame
    loss = np.zeros((NS, F), dtype=np.int8)           # 0 = received, 1 = lost (NULL packet), 2 = cut to the TOC byte
    for i in range(NS):
        mode = rs.randint(4)
        if mode == 1:
            loss[i][rs.rand(F) < 0.1] = 1
        elif mode == 2:
            s0 = int(rs.randint(1, max(2, F - 12)))
            loss[i][s0:s0 + int(rs.randint(1, 12))] = 1
        elif mode == 3:
            loss[i][rs.rand(F) < 0.05] = 2
    return ch, fs, F, cfgs, cut, loss, Fs, dFs, dch, maxb, extra, capmul


def ref_encode(pcm, fs, br, ch, Fs, vbr, cvbr, cx, maxb, force_channels, bandwidth, pin=True):
    """The oracle's encoder with the full settings struct -> (data [F*1276], offs, lens, ranges)."""
    out, offs, lens, ranges = O.encode_stream(pcm, fs, br, ch, Fs=Fs, vbr=vbr, cvbr=cvbr, complexity=cx, max_bytes=maxb,
                                              force_channels=force_channels, bandwidth=bandwidth, pin=pin)
    assert (lens >= 0).all(), lens.min()
    return out, offs, lens, ranges


def main():
    import concentus_b200 as cb
    NB = int(sys.argv[1]) if len(sys.argv) > 1 else 24
    NS = int(sys.argv[2]) if len(sys.argv) > 2 else 48
    SEED = int(sys.argv[3]) if len(sys.argv) > 3 else 1
    WIDE = len(sys.argv) > 4 and sys.argv[4] == "wide"
    ONLY = [int(x) for x in os.environ.get("SWEEP_ONLY", "").split(",") if x]
    L = cb.lib()
    assert L.opus_b200_init(0) == 0
    rs = np.random.RandomState(SEED)
    bad_total, t0 = 0, time.time()
    for b in range(NB):
        ch, fs, F, cfgs, cut, loss, Fs, dFs, dch, maxb, extra, capmul = draw_batch(rs, NS, WIDE)
        dfs = int(fs * dFs // Fs * capmul)             # PCM capacity per packet at the decoder's rate
        if dfs * 25 > dFs * 3:                         # opus_decode conceals at most 120 ms
            dfs = fs * dFs // Fs
        if ONLY and b not in ONLY:
            continue
        pcms = [O.test_signal(F * fs, ch, sd, kind) for (_, _, _, kind, sd) in cfgs]
        enc = cb.EncoderBatch(NS, Fs, ch)
        for i, (br, (vbr, cvbr), cx, _, _) in enumerate(cfgs):
            hp = C.c_void_p(enc.handles[i])
            for req, v in ((cb.OPUS_SET_BITRATE_REQUEST, br), (cb.OPUS_SET_VBR_REQUEST, vbr), (cb.OPUS_SET_VBR_CONSTRAINT_REQUEST, cvbr),
                           (cb.OPUS_SET_COMPLEXITY_REQUEST, cx)):
                assert L.opus_encoder_ctl(hp, req, C.c_int32(v)) == 0
            if extra[i][0]:
                assert L.opus_encoder_ctl(hp, cb.OPUS_SET_FORCE_CHANNELS_REQUEST, C.c_int32(extra[i][0])) == 0
            if extra[i][1]:
                assert L.opus_encoder_ctl(hp, cb.OPUS_SET_BANDWIDTH_REQUEST, C.c_int32(extra[i][1])) == 0
        x = np.stack([p.reshape(F, fs * ch) for p in pcms])
        d1, l1 = enc.encode_span(x[:, :cut].reshape(-1, ch), cut, fs, max_data_bytes=maxb)
        d2, l2 = enc.encode_span(x[:, cut:].reshape(-1, ch), F - cut, fs, max_data_bytes=maxb)
        efr = enc.final_ranges()
        enc.close()
        d = np.concatenate([d1.reshape(NS, cut, maxb), d2.reshape(NS, F - cut, maxb)], axis=1)
        l = np.concatenate([l1.reshape(NS, cut), l2.reshape(NS, F - cut)], axis=1)
        refs = [ref_encode(pcms[i], fs, cfgs[i][0], ch, Fs, cfgs[i][1][0], cfgs[i][1][1], cfgs[i][2], maxb, extra[i][0], extra[i][1], pin=False)
                for i in range(NS)]
        bad_e = []
        for i, (rd, ro, rl, rr) in enumerate(refs):
            rd = rd.reshape(F, 1276)
            ok = np.array_equal(rl, l[i]) and all(np.array_equal(rd[f, :max(rl[f], 0)], d[i, f, :max(rl[f], 0)]) for f in range(F)) and int(rr[-1]) == int(efr[i])
            if not ok:
                bad_e.append((i, cfgs[i]))
        # decode the oracle's packets with the per-stream loss pattern
        lens = np.stack([r[2] for r in refs]).copy()
        lens[loss == 1] = 0
        lens[loss == 2] = 1
        blob = np.concatenate([r[0] for r in refs])
        offs = (np.arange(NS * F, dtype=np.int64) * 1276).reshape(NS, F)
        dec = cb.DecoderBatch(NS, dFs, dch)
        p1, r1 = dec.decode_span(blob, offs[:, :cut].reshape(-1), lens[:, :cut].reshape(-1), cut, dfs)
        p2, r2 = dec.decode_span(blob, offs[:, cut:].reshape(-1), lens[:, cut:].reshape(-1), F - cut, dfs)
        dfr = dec.final_ranges()
        dec.close()
        pcm = np.concatenate([p1.reshape(NS, cut, dfs * dch), p2.reshape(NS, F - cut, dfs * dch)], axis=1)
        rets = np.concatenate([r1.reshape(NS, cut), r2.reshape(NS, F - cut)], axis=1)
        bad_d = []
        for i in range(NS):
            rp, rr, rret = O.decode_stream(blob, offs[i], lens[i], dfs, dch, Fs=dFs, pin=False)
            rp = rp.reshape(F, dfs * dch)
            # what a caller may read: the first ret samples of every row; the rest of a row is compared too (the library
            # zero-fills it, the reference leaves the caller's zero-initialised buffer alone)
            head_ok = all(np.array_equal(rp[f, :max(int(rret[f]), 0) * dch], pcm[i, f, :max(int(rret[f]), 0) * dch]) for f in range(F))
            ok = np.array_equal(rret, rets[i]) and head_ok and np.array_equal(rp, pcm[i]) and int(rr[-1]) == int(dfr[i])
            if not ok:
                fb = np.nonzero((rp != pcm[i]).any(axis=1))[0]
                fr_ = np.nonzero(rret != rets[i])[0]
                bad_d.append((i, cfgs[i], "rets equal", bool(np.array_equal(rret, rets[i])),
                              ("first ret diff", int(fr_[0]), int(rret[fr_[0]]), int(rets[i][fr_[0]]), "len", int(lens[i][fr_[0]])) if fr_.size else "",
                              "decoded samples equal", bool(head_ok), "first bad row", int(fb[0]) if fb.size else -1,
                              "range equal", int(rr[-1]) == int(dfr[i]), "lost", np.nonzero(loss[i])[0][:8].tolist()))
        bad_total += len(bad_e) + len(bad_d)
        print("batch %2d: ch=%d Fs=%5d frame=%4d maxb=%4d F=%3d cut=%3d dec=%5d/%d cap=%4d  encode bad %d  decode bad %d %s" % (b, ch, Fs, fs, maxb, F, cut, dFs, dch, dfs, len(bad_e), len(bad_d),
                                                                                          (bad_e + bad_d)[:2] if (bad_e or bad_d) else ""), flush=True)
    print("parity sweep: %d batches x %d streams, seed %d: %d mismatching streams, %.0f s" % (NB, NS, SEED, bad_total, time.time() - t0))
    sys.exit(1 if bad_total else 0)


if __name__ == "__main__":
    main()

"""Malformed input at batch scale on the GPU (VERDICT r1 item 4; the shape of opus-fix/tests/test_opus_decode.c:279-340, which the
reference runs one packet at a time): more than a million packets — valid ones, random garbage behind a CELT TOC, truncated and
bit-flipped valid packets, TOC-only and lost packets, with the stream's configuration (frame size, bandwidth, channel count)
changing every few packets — through opus_decode_span, every return code, every decoded sample and every final range against the
oracle.  One stream in eight is left untouched: a poisoned neighbour must not change its output.  On the GPU a single
out-of-bounds access would take the whole batch down, so this is also the memory-safety test of the decoder kernels."""
import ctypes as C
import os

import numpy as np
import pytest

import oracle_lib as O

pytestmark = pytest.mark.gpu


def _cb():
    import concentus_b200 as cb
    assert cb.lib().opus_b200_init(0) == 0, "CUDA device required: no CPU fallback exists"
    return cb


def _packet_pool():
    """Valid CELT packets of many configurations: list of (packets list) per base stream."""
    pool = []
    k = 0
    for fs in (120, 240, 480, 960):
        for ch in (1, 2):
            for br, vbr in ((24000, 1), (64000, 0), (160000, 1)):
                x = O.test_signal(fs * 40, ch, 3000 + k, ("music", "tone", "clicks", "noise")[k % 4])
                d, o, l, _ = O.encode_stream(x, fs, br, ch, vbr=vbr, cvbr=0, complexity=(0, 5, 10)[k % 3])
                pool.append([np.ascontiguousarray(d[o[f]:o[f] + l[f]]) for f in range(len(l))])
                k += 1
    return pool


def _make_round(pool, n, F, seed):
    rs = np.random.RandomState(seed)
    chunks, offs, lens = [], np.zeros((n, F), dtype=np.int64), np.zeros((n, F), dtype=np.int32)
    pos = 0
    kinds = np.zeros(6, dtype=np.int64)
    for s in range(n):
        clean = s % 8 == 0
        f = 0
        while f < F:
            base = pool[rs.randint(len(pool))]
            start = rs.randint(len(base))
            run = rs.randint(2, 24)
            for j in range(run):
                if f >= F:
                    break
                p = base[(start + j) % len(base)]
                kind = 0 if clean else int(rs.choice(6, p=[0.45, 0.2, 0.12, 0.12, 0.06, 0.05]))
                if kind == 1:                       # garbage behind a CELT TOC (any frame-count code, any padding / size bytes)
                    m = rs.randint(1, 400)
                    p = rs.randint(0, 256, size=m).astype(np.uint8)
                    p[0] |= 0x80
                elif kind == 2:                     # truncated
                    p = p[:rs.randint(1, len(p) + 1)].copy()
                elif kind == 3:                     # bit flips (the mode bit stays: SILK / hybrid frames are out of scope)
                    p = p.copy()
                    for _ in range(rs.randint(1, 6)):
                        i = rs.randint(len(p))
                        p[i] ^= np.uint8(1 << rs.randint(8))
                    p[0] |= 0x80
                elif kind == 4:                     # TOC only
                    p = p[:1].copy()
                elif kind == 5:                     # lost
                    p = p[:0]
                kinds[kind] += 1
                offs[s, f] = pos
                lens[s, f] = len(p)
                if len(p):
                    chunks.append(p)
                    pos += len(p)
                f += 1
    blob = np.concatenate(chunks + [np.zeros(16, dtype=np.uint8)])
    return blob, offs.reshape(-1), lens.reshape(-1), kinds


@pytest.mark.parametrize("Fs,channels,cap", [(48000, 2, 960), (16000, 1, 320), (24000, 2, 240)])
def test_fuzz_million_packets(Fs, channels, cap):
    cb = _cb()
    pool = _packet_pool()
    threads = os.cpu_count() or 4
    rounds, n, F = (8, 512, 128) if Fs == 48000 else (4, 512, 128)   # 524 K + 2 x 262 K packets over the three decoder configurations
    total = 0
    kinds = np.zeros(6, dtype=np.int64)
    for r in range(rounds):
        blob, offs, lens, kd = _make_round(pool, n, F, 77 * r + Fs // 1000)
        kinds += kd
        dec = cb.DecoderBatch(n, Fs, channels)
        pcm, rets = dec.decode_span(blob, offs, lens, F, cap)
        fr = dec.final_ranges()
        dec.close()
        rpcm, rrng, rret = O.decode_streams(n, F, threads, blob, offs, lens, cap, channels, Fs=Fs, pin=True)
        bad = np.nonzero(rets != rret)[0]
        assert len(bad) == 0, ("return codes", Fs, r, int(bad[0]) // F, int(bad[0]) % F, int(rets[bad[0]]), int(rret[bad[0]]), int(lens[bad[0]]))
        # decoded samples of every packet that produced any
        ours = pcm.reshape(n * F, cap * channels)
        ref = rpcm.reshape(n * F, cap * channels)
        cnt = np.maximum(rret, 0)[:, None] * channels
        mask = np.arange(cap * channels)[None, :] < cnt
        diff = np.nonzero(((ours != ref) & mask).any(axis=1))[0]
        assert len(diff) == 0, ("pcm", Fs, r, int(diff[0]) // F, int(diff[0]) % F, int(rret[diff[0]]), int(lens[diff[0]]))
        assert np.array_equal(fr, rrng.reshape(n, F)[:, -1]), ("final range", Fs, r)
        total += n * F
    assert total >= (520000 if Fs == 48000 else 260000)
    assert (kinds[1:] > 5000).all(), kinds

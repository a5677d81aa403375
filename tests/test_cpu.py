"""CPU-side tests (no GPU needed): the oracle (tests/oracle_lib.py) is pinned against the reference's own golden values and our
committed fixtures; the host simulation of the kernel headers (tests/hostsim, a test tool) is diffed against both; the C ABI
library loads, exports every symbol include/*.h declares and refuses to run without a CUDA device."""
import ctypes as C
import glob
import hashlib
import json
import os
import re
import struct
import subprocess
import sys
import zlib

import numpy as np
import pytest

import oracle_lib as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = sorted(p for p in glob.glob(os.path.join(ROOT, "tests", "golden", "*.npz")) if not os.path.basename(p).startswith("enc_"))
GOLDEN_ENC = sorted(glob.glob(os.path.join(ROOT, "tests", "golden", "enc_*.npz")))
# What the reference's repacketizer / opus_packet_pad returned in the comparisons below (return codes and output bytes, in call
# order), as a digest: recorded when these tests last ran against the reference build, whose results ours matched call for call.
REF_RESULTS = os.path.join(ROOT, "tests", "golden", "reference_results.json")


def _hostsim():
    so = os.path.join(ROOT, "tests", "hostsim", "libhostsim.so")
    src = os.path.join(ROOT, "tests", "hostsim", "hostsim.cpp")
    newest = max(os.path.getmtime(p) for p in glob.glob(os.path.join(ROOT, "concentus_b200", "csrc", "*")) + [src])
    if not os.path.exists(so) or os.path.getmtime(so) < newest:
        subprocess.run(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-Wno-unused-function", "-o", so, src], check=True)
    hs = C.CDLL(so)
    hs.hostsim_decode_stream.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                         C.c_void_p, C.c_void_p]
    hs.hostsim_encode_stream.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p,
                                         C.c_void_p]
    hs.hostsim_encode_stream_pipe.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p,
                                              C.c_void_p, C.c_int]
    hs.hostsim_encode_stream_script.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p,
                                                C.c_int, C.c_void_p, C.c_void_p]
    return hs


def _hostsim_encode(hs, pcm, fs, br, ch, vbr, cvbr, cx, application=O.OPUS_APPLICATION_RESTRICTED_LOWDELAY, max_bytes=1275):
    """The encoder headers compiled for the CPU with a 1-lane team (tests/hostsim).  Returns (packets [F,1276], lens, ranges)."""
    pcm = np.ascontiguousarray(pcm, dtype=np.int16)
    F = pcm.shape[0] // fs
    out = np.zeros((F, 1276), dtype=np.uint8)
    lens = np.zeros(F, dtype=np.int32)
    rng = np.zeros(F, dtype=np.uint32)
    cfg = np.array([application, br, vbr, cvbr, cx, max_bytes, 0, 0], dtype=np.int32)
    hs.hostsim_encode_stream(O.ptr(pcm), F, fs, ch, 48000, O.ptr(cfg), O.ptr(out), 1276, O.ptr(lens), O.ptr(rng))
    return out, lens, rng


class _RefResults:
    """The results the reference returned in one of the comparisons below, in call order, checked as one digest (REF_RESULTS)."""

    def __init__(self, name):
        self.name = name
        self.h = hashlib.blake2b(digest_size=16)

    def add(self, *vals):
        for v in vals:
            self.h.update(np.ascontiguousarray(v).tobytes() if isinstance(v, np.ndarray) else repr(int(v)).encode())
            self.h.update(b"|")

    def check(self):
        want = json.load(open(REF_RESULTS))[self.name]
        assert self.h.hexdigest() == want, "%s: results differ from the reference's (digest %s)" % (self.name, self.h.hexdigest())


def _same_packets(g_data, g_offs, g_lens, out, lens):
    if not np.array_equal(g_lens, lens):
        return False
    return all(np.array_equal(g_data[g_offs[f]:g_offs[f] + g_lens[f]], out[f, :g_lens[f]]) for f in range(len(lens)))


def _hostsim_decode(hs, data, offs, lens, fs, ch):
    F = len(lens)
    pcm = np.zeros((F * fs, ch), dtype=np.int16)
    rng = np.zeros(F, dtype=np.uint32)
    ret = np.zeros(F, dtype=np.int32)
    hs.hostsim_decode_stream(O.ptr(data), O.ptr(np.ascontiguousarray(offs, dtype=np.int64)), O.ptr(np.ascontiguousarray(lens, dtype=np.int32)),
                             F, fs, ch, 48000, O.ptr(pcm), O.ptr(rng), O.ptr(ret))
    return pcm, rng, ret


def _check_against_golden(g, pcm, rng, ret):
    fs = int(g["frame_size"])
    assert np.array_equal(ret, g["rets"])
    assert np.array_equal(rng, g["dec_ranges"])
    crc = np.array([zlib.crc32(pcm[f * fs:(f + 1) * fs].tobytes()) for f in range(len(ret))], dtype=np.uint32)
    assert np.array_equal(crc, g["pcm_crc"])
    assert np.array_equal(pcm[:2 * fs], g["pcm_head"])


# reference KAT: sum of final ranges over all 65,536 3-byte prefixes of a 4-byte packet, CELT configs 16/20/24/28
# (opus-fix/tests/test_opus_decode.c:236-258)
CRES = {16: 116290185, 20: 2172123586, 24: 2172123586, 28: 2172123586}


def cres_packets(cfg):
    i = np.arange(65536, dtype=np.uint32)
    pk = np.stack([np.full(65536, cfg << 3, dtype=np.uint32), i >> 8, i & 255, np.full(65536, 255, dtype=np.uint32)], axis=1)
    data = pk.astype(np.uint8).reshape(-1)
    return data, np.arange(65536, dtype=np.int64) * 4, np.full(65536, 4, dtype=np.int32)


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p)[:-4] for p in GOLDEN])
def test_oracle_reproduces_golden(path):
    g = np.load(path)
    pcm, rng, ret = O.decode_stream(g["data"], g["offs"], g["lens"], int(g["frame_size"]), int(g["channels"]))
    _check_against_golden(g, pcm, rng, ret)
    # encoder and decoder of the reference agree on the final range of every packet (tests/test_opus_encode.c:306)
    assert np.array_equal(g["enc_ranges"], g["dec_ranges"])


@pytest.mark.parametrize("cfg", [16, 28])
def test_oracle_pinned_by_reference_cres_kat(cfg):
    data, offs, lens = cres_packets(cfg)
    _, rng, ret = O.decode_stream(data, offs, lens, 120, 1)
    assert (ret == 120).all()
    assert int(rng.astype(np.uint64).sum() & 0xFFFFFFFF) == CRES[cfg]


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p)[:-4] for p in GOLDEN])
def test_hostsim_matches_golden(path):
    g = np.load(path)
    pcm, rng, ret = _hostsim_decode(_hostsim(), g["data"], g["offs"], g["lens"], int(g["frame_size"]), int(g["channels"]))
    _check_against_golden(g, pcm, rng, ret)


@pytest.mark.parametrize("cfg", [16, 20, 24, 28])
def test_hostsim_cres_kat(cfg):
    data, offs, lens = cres_packets(cfg)
    _, rng, ret = _hostsim_decode(_hostsim(), data, offs, lens, 120, 1)
    assert (ret == 120).all()
    assert int(rng.astype(np.uint64).sum() & 0xFFFFFFFF) == CRES[cfg]


def test_hostsim_vs_oracle_mini_sweep():
    hs = _hostsim()
    seed = 77
    for kind in ("music", "clicks"):
        for ch in (1, 2):
            for fs in (120, 480, 960):
                for br, vbr, cvbr in ((32000, 1, 0), (96000, 0, 0), (256000, 1, 1)):
                    seed += 1
                    x = O.test_signal(24000, ch, seed, kind)
                    d, o, l, _ = O.encode_stream(x, fs, br, vbr=vbr, cvbr=cvbr)
                    rp, rr, rret = O.decode_stream(d, o, l, fs, ch)
                    hp, hr, hret = _hostsim_decode(hs, d, o, l, fs, ch)
                    assert np.array_equal(rret, hret) and np.array_equal(rr, hr) and np.array_equal(rp, hp), (kind, ch, fs, br)


# ---- encoder --------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("path", GOLDEN_ENC, ids=[os.path.basename(p)[:-4] for p in GOLDEN_ENC])
def test_oracle_reproduces_encoder_golden(path):
    g = np.load(path)
    d, o, l, r = O.encode_stream(g["pcm"], int(g["frame_size"]), int(g["bitrate"]), int(g["channels"]), vbr=int(g["vbr"]),
                                 cvbr=int(g["cvbr"]), complexity=int(g["complexity"]))
    assert _same_packets(g["data"], g["offs"], g["lens"], d.reshape(-1, 1276), l)
    assert np.array_equal(r, g["enc_ranges"])
    # and the reference decoder agrees with the encoder on every final range (tests/test_opus_encode.c:306)
    _, dr, _ = O.decode_stream(g["data"], g["offs"], g["lens"], int(g["frame_size"]), int(g["channels"]))
    assert np.array_equal(dr, g["enc_ranges"])


@pytest.mark.parametrize("path", GOLDEN_ENC, ids=[os.path.basename(p)[:-4] for p in GOLDEN_ENC])
def test_hostsim_encoder_matches_golden(path):
    g = np.load(path)
    out, lens, rng = _hostsim_encode(_hostsim(), g["pcm"], int(g["frame_size"]), int(g["bitrate"]), int(g["channels"]), int(g["vbr"]),
                                     int(g["cvbr"]), int(g["complexity"]))
    assert _same_packets(g["data"], g["offs"], g["lens"], out, lens)
    assert np.array_equal(rng, g["enc_ranges"])


def test_hostsim_encoder_vs_oracle_mini_sweep():
    """BASELINE configs[3] in miniature: frame size x channels x bitrate x CBR/VBR/CVBR x complexity x signal kind."""
    hs = _hostsim()
    rs = np.random.RandomState(11)
    cases = [(k, ch, fs, br, m, cx) for k in ("music", "tone", "clicks", "noise") for ch in (1, 2) for fs in (120, 240, 480, 960)
             for br in (32000, 48000, 64000, 96000, 128000, 192000, 256000, 510000) for m in ((0, 0), (1, 0), (1, 1)) for cx in (0, 5, 10)]
    for i in rs.permutation(len(cases))[:120]:
        kind, ch, fs, br, (vbr, cvbr), cx = cases[i]
        x = O.test_signal(24000, ch, 300 + int(i), kind)
        d, o, l, r = O.encode_stream(x, fs, br, ch, vbr=vbr, cvbr=cvbr, complexity=cx)
        out, lens, rng = _hostsim_encode(hs, x, fs, br, ch, vbr, cvbr, cx)
        assert _same_packets(d, o, l, out, lens) and np.array_equal(r, rng), cases[i]


def _hostsim_encode_pipe(hs, pcm, fs, br, ch, vbr, cvbr, cx, Fs=48000, max_bytes=1276, Fc=4):
    """The frame-synchronous encoder pipeline (celt_enc_pipe.cuh) on the CPU: its stages in the kernels' order, chunks of Fc frames."""
    pcm = np.ascontiguousarray(pcm, dtype=np.int16)
    F = pcm.shape[0] // fs
    out = np.zeros((F, 1276), dtype=np.uint8)
    lens = np.zeros(F, dtype=np.int32)
    rng = np.zeros(F, dtype=np.uint32)
    cfg = np.array([O.OPUS_APPLICATION_RESTRICTED_LOWDELAY, br, vbr, cvbr, cx, max_bytes, 0, 0], dtype=np.int32)
    rc = hs.hostsim_encode_stream_pipe(O.ptr(pcm), F, fs, ch, Fs, O.ptr(cfg), O.ptr(out), 1276, O.ptr(lens), O.ptr(rng), Fc)
    return rc, out, lens, rng


@pytest.mark.parametrize("band_mode", [2, 1, 0], ids=["inline_walk", "split_chains", "one_stage"])
def test_hostsim_encoder_pipeline_vs_oracle_mini_sweep(band_mode):
    """The pipeline's slicing of the frame (prepass / front end / head / comb / transform / decide / bands) against the oracle:
    frame size x channels x bitrate x CBR/VBR/CVBR x complexity x signal kind, chunk lengths that do and do not divide the span.
    band_mode: the three forms of the band stage (celt_enc_pipe.cuh K5)."""
    hs = _hostsim()
    hs.hostsim_set_band_mode(band_mode)
    rs = np.random.RandomState(12 + band_mode)
    cases = [(k, ch, fs, br, m, cx) for k in ("music", "tone", "clicks", "noise") for ch in (1, 2) for fs in (120, 240, 480, 960)
             for br in (32000, 48000, 64000, 96000, 128000, 192000, 256000, 510000) for m in ((0, 0), (1, 0), (1, 1)) for cx in (0, 5, 10)]
    for n, i in enumerate(rs.permutation(len(cases))[:(500, 100, 50)[2 - band_mode]]):   # the inline walk is what the GPU runs
        kind, ch, fs, br, (vbr, cvbr), cx = cases[i]
        x = O.test_signal(24000, ch, 500 + int(i), kind)
        d, o, l, r = O.encode_stream(x, fs, br, ch, vbr=vbr, cvbr=cvbr, complexity=cx, max_bytes=1276)
        rc, out, lens, rng = _hostsim_encode_pipe(hs, x, fs, br, ch, vbr, cvbr, cx, Fc=(1, 3, 4, 7, 16)[n % 5])
        assert rc == 0, (cases[i], rc)
        assert _same_packets(d, o, l, out, lens) and np.array_equal(r, rng), cases[i]
    hs.hostsim_set_band_mode(2)


def test_hostsim_encoder_pipeline_long_and_api_rates():
    hs = _hostsim()
    hs.hostsim_set_band_mode(2)
    x = O.test_signal(48000 * 21, 2, 5, "music")
    d, o, l, r = O.encode_stream(x, 960, 96000, 2, vbr=1, cvbr=1, complexity=10, max_bytes=1276)
    rc, out, lens, rng = _hostsim_encode_pipe(hs, x, 960, 96000, 2, 1, 1, 10, Fc=16)
    assert rc == 0 and _same_packets(d, o, l, out, lens) and np.array_equal(r, rng)
    n = 0
    for Fs in (8000, 12000, 16000, 24000):
        for ch in (1, 2):
            for ms in (2.5, 5, 10, 20):
                br, vbr, cvbr = ((24000, 1, 1), (64000, 0, 0), (128000, 1, 0))[n % 3]
                fs = int(Fs * ms / 1000)
                x = O.test_signal(Fs // 2, ch, 70 + n, ("music", "tone", "clicks", "noise")[n % 4])
                n += 1
                d, o, l, r = O.encode_stream(x, fs, br, ch, Fs=Fs, vbr=vbr, cvbr=cvbr, complexity=10, max_bytes=1276)
                rc, out, lens, rng = _hostsim_encode_pipe(hs, x, fs, br, ch, vbr, cvbr, 10, Fs=Fs, Fc=5)
                assert rc == 0 and _same_packets(d, o, l, out, lens) and np.array_equal(r, rng), (Fs, ch, ms, br)
    # low-rate stereo (narrowing, stereo -> mono decision) and a tight byte budget
    for (ch, fs, br, maxb) in ((2, 960, 24000, 1276), (2, 120, 32000, 1276), (2, 480, 36000, 1276), (2, 960, 96000, 120), (1, 240, 510000, 300)):
        x = O.test_signal(48000, ch, 9, "music")
        d, o, l, r = O.encode_stream(x, fs, br, ch, vbr=1, cvbr=0, complexity=10, max_bytes=maxb)
        rc, out, lens, rng = _hostsim_encode_pipe(hs, x, fs, br, ch, 1, 0, 10, max_bytes=maxb, Fc=6)
        assert rc == 0 and _same_packets(d, o, l, out, lens) and np.array_equal(r, rng), (ch, fs, br, maxb)


def test_hostsim_encoder_long_vbr_and_audio_application():
    """The VBR controller settles over ~970 frames (vbr_count); OPUS_APPLICATION_AUDIO adds 4 ms of delay compensation."""
    hs = _hostsim()
    x = O.test_signal(48000 * 21, 2, 5, "music")
    d, o, l, r = O.encode_stream(x, 960, 96000, 2, vbr=1, cvbr=1, complexity=10)
    out, lens, rng = _hostsim_encode(hs, x, 960, 96000, 2, 1, 1, 10)
    assert _same_packets(d, o, l, out, lens) and np.array_equal(r, rng)
    for (ch, fs, br) in ((2, 960, 96000), (2, 240, 128000), (2, 960, 24000)):
        x = O.test_signal(48000, ch, 6, "music")
        d, o, l, r = O.encode_stream(x, fs, br, ch, vbr=1, cvbr=1, complexity=10, application=O.OPUS_APPLICATION_AUDIO)
        assert (d.reshape(-1, 1276)[:, 0] & 0x80).all()      # the reference itself picks CELT-only here
        out, lens, rng = _hostsim_encode(hs, x, fs, br, ch, 1, 1, 10, application=O.OPUS_APPLICATION_AUDIO)
        assert _same_packets(d, o, l, out, lens) and np.array_equal(r, rng), (ch, fs, br)


def test_hostsim_encoder_other_api_rates():
    """Encoder at 8/12/16/24 kHz API rates, both applications, every frame size."""
    hs = _hostsim()
    n = 0
    for Fs in (8000, 12000, 16000, 24000):
        for ch in (1, 2):
            for ms in (2.5, 5, 10, 20):
                br, vbr, cvbr = ((24000, 1, 1), (64000, 0, 0), (128000, 1, 0))[n % 3]
                app = (O.OPUS_APPLICATION_RESTRICTED_LOWDELAY, O.OPUS_APPLICATION_AUDIO)[n % 2]
                fs = int(Fs * ms / 1000)
                x = O.test_signal(Fs // 2, ch, 70 + n, ("music", "tone", "clicks", "noise")[n % 4])
                n += 1
                d, o, l, r = O.encode_stream(x, fs, br, ch, Fs=Fs, vbr=vbr, cvbr=cvbr, complexity=10, application=app, max_bytes=1276)
                if not (d.reshape(-1, 1276)[:, 0] & 0x80).all():
                    continue
                F = x.shape[0] // fs
                out = np.zeros((F, 1276), dtype=np.uint8)
                lens = np.zeros(F, dtype=np.int32)
                rng = np.zeros(F, dtype=np.uint32)
                cfg = np.array([app, br, vbr, cvbr, 10, 1276, 0, 0], dtype=np.int32)
                hs.hostsim_encode_stream(O.ptr(np.ascontiguousarray(x)), F, fs, ch, Fs, O.ptr(cfg), O.ptr(out), 1276, O.ptr(lens), O.ptr(rng))
                assert _same_packets(d, o, l, out, lens) and np.array_equal(r, rng), (Fs, ch, ms, br, app)


def test_hostsim_encoder_long_frames():
    """40 / 60 ms frames through the repacketizer path, VBR and padded CBR, with and without a tight max_data_bytes."""
    hs = _hostsim()
    n = 0
    for Fs in (48000, 16000):
        for ch in (1, 2):
            for ms in (40, 60):
                for maxb in (1276, 400):
                    br, vbr, cvbr = ((24000, 1, 1), (64000, 0, 0), (128000, 1, 0), (510000, 1, 0))[n % 4]
                    fs = Fs * ms // 1000
                    x = O.test_signal(Fs, ch, 170 + n, ("music", "tone", "clicks", "noise")[n % 4])
                    n += 1
                    d, o, l, r = O.encode_stream(x, fs, br, ch, Fs=Fs, vbr=vbr, cvbr=cvbr, complexity=10, max_bytes=maxb)
                    F = x.shape[0] // fs
                    out = np.zeros((F, 1276), dtype=np.uint8)
                    lens = np.zeros(F, dtype=np.int32)
                    rng = np.zeros(F, dtype=np.uint32)
                    cfg = np.array([O.OPUS_APPLICATION_RESTRICTED_LOWDELAY, br, vbr, cvbr, 10, maxb, 0, 0], dtype=np.int32)
                    hs.hostsim_encode_stream(O.ptr(np.ascontiguousarray(x)), F, fs, ch, Fs, O.ptr(cfg), O.ptr(out), 1276, O.ptr(lens), O.ptr(rng))
                    assert _same_packets(d, o, l, out, lens) and np.array_equal(r, rng), (Fs, ch, ms, br, maxb)


def test_hostsim_encoder_ctl_fuzz_vs_oracle():
    """Random ctl changes between frames (bitrate incl. AUTO/MAX, VBR / CVBR, complexity, forced channels, bandwidth caps, loss %,
    LSB depth, prediction, signal type, RESET_STATE) — the reference's own fuzz shape (tests/test_opus_encode.c:236-330), every
    frame size incl. 40 / 60 ms.  Exercises the hysteresis paths (stereo <-> mono, bandwidth steps, CBR <-> VBR)."""
    hs = _hostsim()
    for seed in range(36):
        ch = 1 + seed % 2
        fs = (120, 240, 480, 960, 1920, 2880)[seed % 6]
        F = 100 if fs <= 960 else 30
        x = O.test_signal(fs * F, ch, seed, ("music", "tone", "clicks", "noise")[seed % 4])
        script = O.ctl_script(seed, F, ch)
        rd, rl, rr = O.encode_stream_script(x, fs, ch, script)
        out = np.zeros((F, 1276), dtype=np.uint8)
        lens = np.zeros(F, dtype=np.int32)
        rng = np.zeros(F, dtype=np.uint32)
        cfg = np.array([O.OPUS_APPLICATION_RESTRICTED_LOWDELAY, 64000, 1, 1, 10, 1276, 0, 0], dtype=np.int32)
        hs.hostsim_encode_stream_script(O.ptr(np.ascontiguousarray(x)), F, fs, ch, 48000, O.ptr(cfg), O.ptr(np.ascontiguousarray(script)), 2,
                                        O.ptr(out), 1276, O.ptr(lens), O.ptr(rng))
        assert np.array_equal(rl, lens), (seed, int(np.nonzero(rl != lens)[0][0]))
        assert np.array_equal(rr, rng), seed
        for f in range(F):
            assert np.array_equal(rd[f, :rl[f]], out[f, :rl[f]]), (seed, f)


def test_encoder_host_api_ctl_and_padding():
    """Host-side half of the encoder C ABI: sizes, init argument checks, ctl set/get round trips and range checks
    (opus-fix/tests/test_opus_api.c encoder section), opus_packet_pad / unpad against the reference's."""
    import concentus_b200 as cb
    L = cb.lib()
    assert L.opus_encoder_get_size(0) == 0 and L.opus_encoder_get_size(3) == 0
    for ch in (1, 2):
        assert 2048 < L.opus_encoder_get_size(ch) <= (1 << 17)
    err = C.c_int(0)
    assert L.opus_encoder_create(48000, 2, 1234, C.byref(err)) is None and err.value == cb.OPUS_BAD_ARG
    assert L.opus_encoder_create(48000, 3, cb.OPUS_APPLICATION_AUDIO, C.byref(err)) is None and err.value == cb.OPUS_BAD_ARG
    h = L.opus_encoder_create(48000, 2, cb.OPUS_APPLICATION_RESTRICTED_LOWDELAY, C.byref(err))
    assert h and err.value == 0
    hp = C.c_void_p(h)
    v = C.c_int32(0)
    for (setr, getr, good, bad) in ((4002, 4003, 96000, 0), (4010, 4011, 7, 11), (4006, 4007, 0, 2), (4020, 4021, 0, 2), (4022, 4023, 1, 3),
                                    (4004, 4005, 1104, 1100), (4014, 4015, 20, 101), (4036, 4037, 16, 7), (4042, 4043, 1, 2), (4024, 4025, 3002, 5)):
        assert L.opus_encoder_ctl(hp, setr, C.c_int32(good)) == 0, setr
        assert L.opus_encoder_ctl(hp, getr, C.byref(v)) == 0 and v.value == good, getr
        assert L.opus_encoder_ctl(hp, setr, C.c_int32(bad)) == cb.OPUS_BAD_ARG, setr
        assert L.opus_encoder_ctl(hp, getr, None) == cb.OPUS_BAD_ARG
    assert L.opus_encoder_ctl(hp, 4002, C.c_int32(5000000)) == 0 and L.opus_encoder_ctl(hp, 4003, C.byref(v)) == 0 and v.value == 600000
    assert L.opus_encoder_ctl(hp, 4027, C.byref(v)) == 0 and v.value == 120                      # lookahead, restricted low delay
    assert L.opus_encoder_ctl(hp, 4029, C.byref(v)) == 0 and v.value == 48000
    assert L.opus_encoder_ctl(hp, 4000, C.c_int32(cb.OPUS_APPLICATION_AUDIO)) == 0                # allowed before the first frame
    assert L.opus_encoder_ctl(hp, 4027, C.byref(v)) == 0 and v.value == 120 + 192
    assert L.opus_encoder_ctl(hp, 31337, C.c_int32(0)) == cb.OPUS_UNIMPLEMENTED
    before = C.string_at(h, L.opus_encoder_get_size(2))
    assert L.opus_encoder_ctl(hp, cb.OPUS_RESET_STATE) == 0
    L.opus_encoder_destroy(hp)
    assert len(before) == L.opus_encoder_get_size(2)
    # padding: a code-0 packet grown to every size up to +600 bytes, and back
    pk = np.zeros(1276, dtype=np.uint8)
    pk[:40] = np.arange(40) + 0xF8
    ref = _RefResults("opus_packet_pad_code0")
    for new_len in (40, 41, 42, 100, 295, 296, 297, 640):
        a = pk.copy()
        assert L.opus_packet_pad(O.ptr(a), 40, new_len) == 0
        ref.add(a[:new_len])
        assert L.opus_packet_unpad(O.ptr(a), new_len) == 40 and np.array_equal(a[:40], pk[:40])
    assert L.opus_packet_pad(O.ptr(pk), 40, 39) == cb.OPUS_BAD_ARG
    ref.check()                                    # the padded packets are the reference's, byte for byte


@pytest.mark.parametrize("pattern", ["single", "burst", "random", "toc_only", "start_lost"])
def test_hostsim_packet_loss_concealment_vs_oracle(pattern):
    """celt_decode_lost (pitch-based and, after 5 losses, noise-based) through the host simulation of the stage-B code."""
    hs = _hostsim()
    cases = [("music", 2, 960, 64000), ("tone", 2, 960, 96000), ("tone", 1, 480, 48000), ("clicks", 2, 240, 128000), ("music", 1, 120, 64000)]
    for k, (kind, ch, fs, br) in enumerate(cases):
        x = O.test_signal(48000, ch, 40 + k, kind)
        d, o, l, _ = O.encode_stream(x, fs, br, ch, vbr=1, cvbr=0)
        d, o = O.pack(d, o, l)
        l = l.copy()
        F = len(l)
        rs = np.random.RandomState(k)
        if pattern == "single":
            l[10::17] = 0
        elif pattern == "burst":
            for f in range(12, F, 40):
                l[f:f + 8] = 0
        elif pattern == "random":
            l[rs.rand(F) < 0.2] = 0
        elif pattern == "toc_only":
            l[9::13] = 1
        else:
            l[:3] = 0
        rp, rr, rret = O.decode_stream(d, o, l, fs, ch)
        hp, hr, hret = _hostsim_decode(hs, d, o, l, fs, ch)
        assert np.array_equal(rret, hret) and np.array_equal(rr, hr) and np.array_equal(rp, hp), (pattern, kind, ch, fs)


def test_hostsim_garbage_packets_do_not_crash_and_match_oracle():
    hs = _hostsim()
    rs = np.random.RandomState(5)
    F = 400
    lens = rs.randint(3, 60, size=F).astype(np.int32)   # >= 2 payload bytes: a 1-byte payload is a PLC frame (SURVEY 8f, next)
    offs = np.zeros(F, dtype=np.int64)
    offs[1:] = np.cumsum(lens[:-1])
    data = rs.randint(0, 256, size=int(lens.sum())).astype(np.uint8)
    # CELT-only, code 0, 2.5..20 ms, mono/stereo TOCs
    for f in range(F):
        data[offs[f]] = 0x80 | (rs.randint(0, 16) << 3) | (rs.randint(0, 2) << 2)
    hp, hr, hret = _hostsim_decode(hs, data, offs, lens, 960, 2)
    assert ((hret > 0) | (hret == -3)).all()    # garbage may overrun its bit budget: OPUS_INTERNAL_ERROR like the reference
    rp, rr, rret = O.decode_stream(data, offs, lens, 960, 2)
    assert np.array_equal(rret, hret) and np.array_equal(rr, hr)
    for f in range(F):
        n = max(int(hret[f]), 0)
        assert np.array_equal(rp[f * 960:f * 960 + n], hp[f * 960:f * 960 + n]), f


def _declared_symbols():
    names = set()
    for h in glob.glob(os.path.join(ROOT, "include", "*.h")):
        txt = re.sub(r"/\*.*?\*/", "", open(h).read(), flags=re.S)
        for m in re.finditer(r"\b(opus_[a-z0-9_]+)\s*\(", txt):
            names.add(m.group(1))
    return sorted(names)


def test_cabi_library_loads_and_exports_every_declared_symbol():
    import concentus_b200 as cb
    L = cb.lib()
    syms = _declared_symbols()
    assert len(syms) >= 20
    for s in syms:
        assert hasattr(L, s), "include/*.h declares %s but the library does not export it" % s
    assert b"-fixed" in L.opus_get_version_string()
    assert L.opus_strerror(-4) == b"corrupted stream"


def test_host_side_packet_helpers_and_state_block():
    import concentus_b200 as cb
    L = cb.lib()
    toc = np.array([0xFC, 1, 2, 3], dtype=np.uint8)
    assert L.opus_packet_get_bandwidth(O.ptr(toc)) == 1105
    assert L.opus_packet_get_nb_channels(O.ptr(toc)) == 2
    assert L.opus_packet_get_samples_per_frame(O.ptr(toc), 48000) == 960
    assert L.opus_packet_get_nb_frames(O.ptr(toc), 4) == 1
    assert L.opus_packet_get_nb_samples(O.ptr(toc), 4, 48000) == 960
    for ch in (1, 2):
        n = L.opus_decoder_get_size(ch)
        assert 2048 < n <= (1 << 16)          # bounds checked by opus-fix/tests/test_opus_api.c:106
    assert L.opus_decoder_get_size(0) == 0 and L.opus_decoder_get_size(3) == 0
    err = C.c_int(0)
    h = L.opus_decoder_create(48000, 2, C.byref(err))
    assert h and err.value == 0
    v = C.c_int32(0)
    assert L.opus_decoder_ctl(C.c_void_p(h), cb.OPUS_GET_SAMPLE_RATE_REQUEST, C.byref(v)) == 0 and v.value == 48000
    assert L.opus_decoder_ctl(C.c_void_p(h), cb.OPUS_SET_GAIN_REQUEST, C.c_int32(40000)) == cb.OPUS_BAD_ARG
    assert L.opus_decoder_ctl(C.c_void_p(h), 12345) == cb.OPUS_UNIMPLEMENTED
    assert L.opus_decoder_ctl(C.c_void_p(h), cb.OPUS_RESET_STATE) == 0
    L.opus_decoder_destroy(C.c_void_p(h))


def test_product_fails_loudly_without_cuda():
    """No CPU fallback: on a box without a GPU every codec call must return OPUS_INTERNAL_ERROR."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    code = ("import ctypes as C, numpy as np, concentus_b200 as cb; L=cb.lib(); e=C.c_int(0);"
            "h=L.opus_decoder_create(48000,2,C.byref(e)); p=np.array([0xFC,1,2,3],dtype=np.uint8); o=np.zeros(1920,dtype=np.int16);"
            "r=L.opus_decode(C.c_void_p(h), p.ctypes.data_as(C.c_void_p), 4, o.ctypes.data_as(C.c_void_p), 960, 0); print(r, L.opus_b200_init(0))")
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=ROOT)
    assert out.stdout.split() == ["-3", "-3"], (out.stdout, out.stderr)
    code = ("import ctypes as C, numpy as np, concentus_b200 as cb; L=cb.lib(); e=C.c_int(0);"
            "h=L.opus_encoder_create(48000,2,2051,C.byref(e)); x=np.zeros(1920,dtype=np.int16); o=np.zeros(1276,dtype=np.uint8);"
            "r=L.opus_encode(C.c_void_p(h), x.ctypes.data_as(C.c_void_p), 960, o.ctypes.data_as(C.c_void_p), 1276); print(r)")
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=ROOT)
    assert out.stdout.split() == ["-3"], (out.stdout, out.stderr)


def _gloo_worker(rank, world, port, q):
    import torch
    import torch.distributed as dist
    from concentus_b200.shard import shard_range
    dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%d" % port, rank=rank, world_size=world)
    b, e = shard_range(4099, world, rank)
    t = torch.tensor([e - b, b, e], dtype=torch.int64)
    out = [torch.zeros(3, dtype=torch.int64) for _ in range(world)]
    dist.all_gather(out, t)
    ms = torch.tensor([10.0 + rank])
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)        # the timing reduction bench.py does
    dist.barrier()
    if rank == 0:
        q.put(([o.tolist() for o in out], float(ms.item())))
    dist.destroy_process_group()


def test_stream_sharding_world_size_2_gloo():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 2000)
    ps = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in ps:
        p.start()
    res, ms = q.get(timeout=120)
    for p in ps:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert res[0][1] == 0 and res[0][2] == res[1][1] and res[1][2] == 4099      # contiguous, disjoint, complete
    assert res[0][0] + res[1][0] == 4099 and abs(res[0][0] - res[1][0]) <= 1
    assert ms == 11.0


# ---- the .bit container (SURVEY.md §8f rank 4): pinned on files written by the reference's own opus_demo -----------------------

def _opus_demo_file(ch, fs, br):
    """tests/golden/opus_demo_*.bit: the file `opus_demo -e restricted-lowdelay 48000 <ch> <br> -framesize <ms>` of the reference
    wrote for test_signal(48000, ch, 77 + ch, "music")."""
    ms = {120: "2.5", 240: "5", 480: "10", 960: "20"}[fs]
    return os.path.join(ROOT, "tests", "golden", "opus_demo_%dch_%sms_%dk.bit" % (ch, ms, br // 1000))


@pytest.mark.parametrize("ch,fs,br", [(2, 960, 64000), (1, 480, 48000), (2, 120, 128000)])
def test_bit_container_reads_what_opus_demo_writes(tmp_path, ch, fs, br):
    """opus_demo -e (src/opus_demo.c:748-760) wrote the file; our reader must return exactly the packets and final ranges the
    oracle's encoder produces for the same input, and our writer must reproduce the file byte for byte."""
    from concentus_b200 import bitfile
    pcm = O.test_signal(48000, ch, 77 + ch, "music")
    bit = _opus_demo_file(ch, fs, br)
    data, offs, lens, ranges = bitfile.read_bit(str(bit))
    # opus_demo codes one extra all-zero frame when the input ends on a frame boundary (src/opus_demo.c:672-690)
    x = np.concatenate([pcm, np.zeros((fs, ch), dtype=np.int16)])
    rd, ro, rl, rr = O.encode_stream(x, fs, br, ch, vbr=1, cvbr=0, complexity=10, max_bytes=1500)
    F = len(rl)
    assert len(lens) == F and np.array_equal(lens, rl)
    assert np.array_equal(ranges, rr)
    for f in range(F):
        assert np.array_equal(data[offs[f]:offs[f] + lens[f]], rd[ro[f]:ro[f] + rl[f]]), f
    out = tmp_path / "ours.bit"
    bitfile.write_bit(str(out), data, offs, lens, ranges)
    assert open(out, "rb").read() == open(bit, "rb").read()


def test_bit_container_edge_cases(tmp_path):
    from concentus_b200 import bitfile
    empty = tmp_path / "empty.bit"
    empty.write_bytes(b"")
    d, o, l, r = bitfile.read_bit(str(empty))
    assert len(l) == 0 and len(o) == 0 and len(r) == 0
    # a lost packet (length 0) and a truncated tail: the reader stops where opus_demo would (short read, :665-670)
    pk = bytes([0xFC, 1, 2, 3])
    good = struct.pack(">II", 4, 0x12345678) + pk + struct.pack(">II", 0, 0) + struct.pack(">II", 4, 7) + pk
    f = tmp_path / "trunc.bit"
    f.write_bytes(good + struct.pack(">II", 100, 1) + b"\x01\x02")
    d, o, l, r = bitfile.read_bit(str(f))
    assert l.tolist() == [4, 0, 4] and r.tolist() == [0x12345678, 0, 7]
    assert bytes(d[o[2]:o[2] + 4]) == pk
    # an absurd length field ends the stream as well (opus_demo: "Invalid payload length")
    g = tmp_path / "bad.bit"
    g.write_bytes(good + struct.pack(">II", 1 << 20, 1))
    assert bitfile.read_bit(str(g))[2].tolist() == [4, 0, 4]


def test_hostsim_call_boundaries_with_loss_runs():
    """The decoder headers under explicit call boundaries (hostsim_decode_stream_calls): stage A of a call starts from the
    call-start snapshot (CbCallCtx) and tracks seed / loss streak through lost packets; calls that begin inside a burst, right
    after one, and with TOC-only packets."""
    hs = _hostsim()
    hs.hostsim_decode_stream_calls.argtypes = [C.c_void_p] * 3 + [C.c_int] * 4 + [C.c_void_p] * 3 + [C.c_void_p, C.c_int]
    for k, (ch, fs, br, cuts) in enumerate(((2, 480, 96000, [83, 200]), (2, 240, 40000, [50, 51, 120, 200]), (1, 960, 64000, [7, 30, 31, 100]))):
        x = O.test_signal(fs * cuts[-1], ch, 600 + k, ("music", "clicks", "tone")[k])
        d, o, l, _ = O.encode_stream(x, fs, br, ch, vbr=1, cvbr=0)
        d, o = O.pack(d, o, l)
        l = l.copy()
        F = len(l)
        c0 = cuts[0]
        l[c0 - (k % 2):c0 + 11] = 0          # a burst that starts at / just before the first boundary and outlasts pitch-based PLC
        l[c0 + 30] = 1                        # TOC-only
        rp, rr, rret = O.decode_stream(d, o, l, fs, ch)
        pcm = np.zeros((F * fs, ch), dtype=np.int16)
        rng = np.zeros(F, dtype=np.uint32)
        ret = np.zeros(F, dtype=np.int32)
        b = np.array(cuts, dtype=np.int32)
        hs.hostsim_decode_stream_calls(O.ptr(d), O.ptr(np.ascontiguousarray(o, dtype=np.int64)), O.ptr(np.ascontiguousarray(l, dtype=np.int32)),
                                       F, fs, ch, 48000, O.ptr(pcm), O.ptr(rng), O.ptr(ret), O.ptr(b), len(cuts))
        assert np.array_equal(ret, rret) and np.array_equal(rng, rr), (ch, fs)
        bad = np.nonzero((rp.reshape(F, -1) != pcm.reshape(F, -1)).any(axis=1))[0]
        assert bad.size == 0, (ch, fs, int(bad[0]))


def test_hostsim_random_wide_sweep():
    """A small slice of tools/hostsim_sweep.py in the CPU suite: random batches in wide mode (API rates, 40 / 60 ms frames,
    starved max_data_bytes, forced channels / bandwidth, decoder rate / channels / PCM capacity differing from the stream's,
    random / burst / TOC-only loss, a call boundary at a random packet) through the kernel headers with 1-lane teams."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import hostsim_sweep as HS
    import parity_sweep as PS
    rs = np.random.RandomState(2024)
    bad = []
    for b in range(10):
        ch, fs, F, cfgs, cut, loss, Fs, dFs, dch, maxb, extra, capmul = PS.draw_batch(rs, 6, True)
        for i in range(6):
            r = HS.one_stream((b, i, ch, fs, F, cfgs[i], cut, loss[i], Fs, dFs, dch, maxb, extra[i], capmul))
            if not (r[2] and r[3]):
                bad.append(r)
    assert not bad, bad[:3]


def test_repacketizer_and_pad_unpad_match_the_reference():
    """opus_repacketizer_* and opus_packet_pad / opus_packet_unpad for packets of every frame-count code (host code of the library,
    opus-fix/src/repacketizer.c:37-273): same return codes and bytes as the reference on random merges, splits and paddings."""
    import concentus_b200 as cb
    L = cb.lib()
    L.opus_repacketizer_create.restype = C.c_void_p
    L.opus_repacketizer_init.restype = C.c_void_p
    L.opus_repacketizer_init.argtypes = [C.c_void_p]
    L.opus_repacketizer_destroy.argtypes = [C.c_void_p]
    L.opus_repacketizer_cat.argtypes = [C.c_void_p, C.c_void_p, C.c_int32]
    L.opus_repacketizer_get_nb_frames.argtypes = [C.c_void_p]
    L.opus_repacketizer_out.argtypes = [C.c_void_p, C.c_void_p, C.c_int32]
    L.opus_repacketizer_out_range.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int32]
    L.opus_packet_pad.argtypes = [C.c_void_p, C.c_int32, C.c_int32]
    L.opus_packet_unpad.argtypes = [C.c_void_p, C.c_int32]
    assert L.opus_repacketizer_get_size() > 0
    ref = _RefResults("repacketizer_pad_unpad")
    rs = np.random.RandomState(5)
    rp_l = L.opus_repacketizer_create()
    n_multi = 0
    for trial in range(60):
        fs = (120, 240, 480, 960)[trial % 4]
        ch = 1 + (trial // 4) % 2
        vbr = (trial // 8) % 2
        x = O.test_signal(fs * 12, ch, 900 + trial, ("music", "tone", "clicks", "noise")[trial % 4])
        d, o, l, _ = O.encode_stream(x, fs, (24000, 64000, 128000)[trial % 3], ch, vbr=vbr, cvbr=0)
        pk = [np.ascontiguousarray(d[o[f]:o[f] + l[f]]) for f in range(len(l))]
        if trial % 5 == 4:
            pk[3] = np.ascontiguousarray(pk[3][:1])            # a TOC-only packet among them
        if trial % 7 == 6:
            pk[2] = pk[2].copy(); pk[2][0] ^= 0x08             # a packet of another configuration: must be refused
        L.opus_repacketizer_init(rp_l)
        ncat = int(rs.randint(1, 9))
        for k in range(ncat):
            ref.add(L.opus_repacketizer_cat(rp_l, O.ptr(pk[k]), len(pk[k])))
        nf = L.opus_repacketizer_get_nb_frames(rp_l)
        ref.add(nf)
        for maxlen in (3000, int(rs.randint(1, 600)), 1):
            ol = np.zeros(3000, dtype=np.uint8)
            a = L.opus_repacketizer_out(rp_l, O.ptr(ol), maxlen)
            ref.add(a, ol[:max(a, 0)])
            if nf >= 1:
                lo = int(rs.randint(0, nf)); hi = int(rs.randint(lo, nf + 2))
                a = L.opus_repacketizer_out_range(rp_l, lo, hi, O.ptr(ol), maxlen)
                ref.add(a, ol[:max(a, 0)])
        # pad / unpad of the merged (multi-frame) packet, in place
        ol = np.zeros(4000, dtype=np.uint8)
        n = L.opus_repacketizer_out(rp_l, O.ptr(ol), 3000)
        if n > 0:
            n_multi += nf > 1
            for new_len in (n, n + 1, n + 2, n + int(rs.randint(3, 700)), n - 1):
                bl = ol.copy()
                a = L.opus_packet_pad(O.ptr(bl), n, new_len)
                ref.add(a)
                if a == 0:
                    ref.add(bl[:new_len])
                    a = L.opus_packet_unpad(O.ptr(bl), new_len)
                    ref.add(a, bl[:max(a, 0)])
    assert n_multi >= 30
    for bad in (0, -3):
        buf = np.zeros(16, dtype=np.uint8)
        ref.add(L.opus_packet_pad(O.ptr(buf), bad, 8), L.opus_packet_unpad(O.ptr(buf), bad))
    L.opus_repacketizer_destroy(rp_l)
    ref.check()


def test_public_header_compiles_reference_style_ctl_calls(tmp_path):
    """include/opus_b200.h carries the reference's OPUS_SET_* / OPUS_GET_* convenience macros (opus_defines.h:107-122), so a source
    written against opus.h compiles against it unchanged (VERDICT r1: the macros were missing)."""
    src = tmp_path / "ctl.c"
    src.write_text('''
#include "opus_b200.h"
int f(OpusEncoder *e, OpusDecoder *d) {
    opus_int32 v; opus_uint32 r; int rc = 0;
    rc |= opus_encoder_ctl(e, OPUS_SET_BITRATE(64000));
    rc |= opus_encoder_ctl(e, OPUS_SET_VBR(1));
    rc |= opus_encoder_ctl(e, OPUS_SET_COMPLEXITY(10));
    rc |= opus_encoder_ctl(e, OPUS_GET_LOOKAHEAD(&v));
    rc |= opus_encoder_ctl(e, OPUS_GET_FINAL_RANGE(&r));
    rc |= opus_encoder_ctl(e, OPUS_SET_LFE(0));
    rc |= opus_decoder_ctl(d, OPUS_SET_GAIN(0));
    rc |= opus_decoder_ctl(d, OPUS_GET_LAST_PACKET_DURATION(&v));
    return rc;
}
''')
    r = subprocess.run(["gcc", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-c", str(src), "-o", str(tmp_path / "ctl.o")],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr

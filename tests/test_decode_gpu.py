"""GPU parity: CUDA decode (through the C ABI of libconcentus_b200.so) vs the oracle (tests/oracle_lib.py: the results of the
unmodified opus-fix build), PCM sample-for-sample, final range per packet and return code per packet."""
import ctypes as C
import os
import zlib

import numpy as np
import pytest

import oracle_lib as O

pytestmark = pytest.mark.gpu
# What the reference decoder returned in test_decoder_gain_ctl / test_decoder_getters_and_reset_per_packet (oracle/ref_harness.c
# ref_decode_stream_gain / ref_decode_stream_info on the same packets): per packet the return code, final range, CRC-32 of the
# decoded samples and the getters' values.
DECODER_CTL = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "decoder", "ctl.npz")


def _row_crc(rows):
    return np.array([zlib.crc32(np.ascontiguousarray(r).tobytes()) for r in rows], dtype=np.uint32)


def _cb():
    import concentus_b200 as cb
    assert cb.lib().opus_b200_init(0) == 0, "CUDA device required: no CPU fallback exists"
    return cb


def _make_streams(cfgs, nsec):
    """cfgs: list of (kind, channels_in, frame_size, bitrate, vbr, cvbr, seed); all decoded by `channels`-ch decoders."""
    datas, lens_all, offs_all = [], [], []
    base = 0
    for (kind, ch, fs, br, vbr, cvbr, seed) in cfgs:
        pcm = O.test_signal(48000 * nsec, ch, seed, kind)
        d, o, l, _ = O.encode_stream(pcm, fs, br, vbr=vbr, cvbr=cvbr)
        d, o = O.pack(d, o, l)
        datas.append(d)
        offs_all.append(o + base)
        lens_all.append(l)
        base += len(d)
    return np.concatenate(datas), np.concatenate(offs_all), np.concatenate(lens_all)


def _check(cfgs, dec_channels, frame_size, nsec=1):
    cb = _cb()
    data, offs, lens = _make_streams(cfgs, nsec)
    n = len(cfgs)
    F = len(lens) // n
    dec = cb.DecoderBatch(n, 48000, dec_channels)
    # decode in two spans to exercise state residency across launches
    F1 = F // 2
    idx = np.arange(n * F).reshape(n, F)
    pcm = np.zeros((n, F, frame_size * dec_channels), dtype=np.int16)
    rets = np.zeros((n, F), dtype=np.int32)
    for (a, b) in ((0, F1), (F1, F)):
        sel = idx[:, a:b].reshape(-1)
        p, r = dec.decode_span(data, offs[sel], lens[sel], b - a, frame_size)
        pcm[:, a:b] = p.reshape(n, b - a, -1)
        rets[:, a:b] = r.reshape(n, b - a)
    fr = dec.final_ranges()
    dec.close()
    for s in range(n):
        sel = idx[s]
        rp, rr, rret = O.decode_stream(data, offs[sel], lens[sel], frame_size, dec_channels)
        assert np.array_equal(rret, rets[s]), ("ret", cfgs[s])
        bad = np.nonzero((rp.reshape(F, -1) != pcm[s]).any(axis=1))[0]
        assert bad.size == 0, ("pcm mismatch", cfgs[s], "first bad frame", int(bad[0]))
        assert int(rr[-1]) == int(fr[s]), ("final range", cfgs[s])


@pytest.mark.parametrize("fs", [120, 240, 480, 960])
@pytest.mark.parametrize("ch", [1, 2])
def test_sweep_framesize_channels(fs, ch):
    cfgs = []
    seed = 100 * ch + fs
    for kind in ("music", "tone", "clicks", "noise"):
        for br in (32000, 64000, 128000, 510000):
            for (vbr, cvbr) in ((1, 0), (0, 0), (1, 1)):
                cfgs.append((kind, ch, fs, br, vbr, cvbr, seed))
                seed += 1
    _check(cfgs, ch, fs, nsec=1)


def test_mono_stream_into_stereo_decoder_and_back():
    cfgs = [("music", 1, 960, 48000, 1, 0, 5), ("tone", 1, 480, 64000, 0, 0, 6)]
    _check([cfgs[0]], 2, 960)
    _check([cfgs[1]], 2, 480)
    cfgs2 = [("music", 2, 960, 96000, 1, 0, 7)]
    _check(cfgs2, 1, 960)


def test_scalar_api_matches_oracle_and_state_is_memcpyable():
    cb = _cb()
    L = cb.lib()
    pcm_in = O.test_signal(48000, 2, 11, "music")
    d, o, l, _ = O.encode_stream(pcm_in, 960, 64000)
    rp, rr, _ = O.decode_stream(d, o, l, 960, 2)
    err = C.c_int(0)
    h = L.opus_decoder_create(48000, 2, C.byref(err))
    assert h and err.value == 0
    size = L.opus_decoder_get_size(2)
    out = np.zeros((960, 2), dtype=np.int16)
    v = C.c_uint32(0)
    for f in range(len(l)):
        if f == 20:
            # clone the state block with memcpy and continue on the clone (tests/test_opus_decode.c:84-95)
            buf = C.create_string_buffer(size)
            C.memmove(buf, h, size)
            L.opus_decoder_destroy(C.c_void_p(h))
            h = C.cast(buf, C.c_void_p).value
        pkt = d[o[f]:o[f] + l[f]].copy()
        r = L.opus_decode(C.c_void_p(h), O.ptr(pkt), int(l[f]), O.ptr(out), 960, 0)
        assert r == 960
        assert np.array_equal(out, rp[f * 960:(f + 1) * 960]), f
        L.opus_decoder_ctl(C.c_void_p(h), cb.OPUS_GET_FINAL_RANGE_REQUEST, C.byref(v))
        assert v.value == int(rr[f])


def test_error_codes_and_scope_edge():
    cb = _cb()
    L = cb.lib()
    err = C.c_int(0)
    assert not L.opus_decoder_create(44100, 2, C.byref(err)) and err.value == cb.OPUS_BAD_ARG
    assert L.opus_decoder_get_size(3) == 0
    h = L.opus_decoder_create(48000, 2, C.byref(err))
    out = np.zeros((5760, 2), dtype=np.int16)
    silk = np.array([0x08, 1, 2, 3], dtype=np.uint8)       # SILK-only TOC: outside this engine
    assert L.opus_decode(C.c_void_p(h), O.ptr(silk), 4, O.ptr(out), 960, 0) == cb.OPUS_UNIMPLEMENTED
    celt = np.array([0xFC, 1, 2, 3], dtype=np.uint8)
    assert L.opus_decode(C.c_void_p(h), O.ptr(celt), 4, O.ptr(out), 120, 0) == cb.OPUS_BUFFER_TOO_SMALL
    assert L.opus_decode(C.c_void_p(h), O.ptr(celt), 4, O.ptr(out), 0, 0) == cb.OPUS_BAD_ARG
    bad = np.array([0xFD, 1, 2, 3], dtype=np.uint8)        # code 1 with odd payload
    assert L.opus_decode(C.c_void_p(h), O.ptr(bad), 4, O.ptr(out), 5760, 0) == cb.OPUS_INVALID_PACKET
    # before any packet, concealment returns zeros (opus_decoder.c:265-272)
    out[:] = 7
    assert L.opus_decode(C.c_void_p(h), None, 0, O.ptr(out), 960, 0) == 960
    assert not out[:960].any()
    L.opus_decoder_destroy(C.c_void_p(h))


def _lossy(lens, pattern, seed):
    """Mark packets lost (len 0 -> opus_decode(NULL)) or cut to a bare TOC (len 1 -> PLC as well, opus_decoder.c:246-252)."""
    l = lens.copy()
    F = len(l)
    rs = np.random.RandomState(seed)
    if pattern == "single":
        l[10::17] = 0
    elif pattern == "burst":                     # 8 in a row: pitch-based for 5 frames, then noise-based (celt_decoder.c:446)
        for f in range(12, F, 40):
            l[f:f + 8] = 0
    elif pattern == "random":
        l[rs.rand(F) < 0.2] = 0
    elif pattern == "toc_only":
        l[9::13] = 1
    elif pattern == "start_lost":
        l[:3] = 0
    return l


@pytest.mark.parametrize("pattern", ["single", "burst", "random", "toc_only", "start_lost"])
def test_packet_loss_concealment(pattern):
    """celt_decode_lost (celt_decoder.c:415-711) through the batch API: NULL / TOC-only packets inside received streams, the
    way tests/test_opus_decode.c:125-132 and opus_demo -loss drive it.  PCM, return codes and final ranges vs the oracle."""
    cb = _cb()
    cases = [("music", 2, 960, 64000), ("tone", 2, 960, 96000), ("tone", 1, 480, 48000), ("clicks", 2, 240, 128000),
             ("music", 1, 120, 64000), ("noise", 2, 960, 128000)]
    for k, (kind, ch, fs, br) in enumerate(cases):
        x = O.test_signal(48000, ch, 40 + k, kind)
        d, o, l, _ = O.encode_stream(x, fs, br, ch, vbr=1, cvbr=0)
        d, o = O.pack(d, o, l)
        l = _lossy(l, pattern, k)
        F = len(l)
        rp, rr, rret = O.decode_stream(d, o, l, fs, ch)
        dec = cb.DecoderBatch(1, 48000, ch)
        F1 = F // 3                                   # two launches: the concealment state crosses a launch boundary
        p1, r1 = dec.decode_span(d, o[:F1], l[:F1], F1, fs)
        p2, r2 = dec.decode_span(d, o[F1:], l[F1:], F - F1, fs)
        fr = dec.final_ranges()
        dec.close()
        assert np.array_equal(np.concatenate([r1, r2]), rret), (pattern, kind, ch, fs)
        got = np.concatenate([p1, p2])
        bad = np.nonzero((rp.reshape(F, -1) != got.reshape(F, -1)).any(axis=1))[0]
        assert bad.size == 0, (pattern, kind, ch, fs, "first bad frame", int(bad[0]), "lost", np.nonzero(l <= 1)[0][:6].tolist())
        assert int(rr[-1]) == int(fr[0])


def test_scalar_api_null_packet_and_fec_flag():
    """opus_decode(st, NULL, 0, ...) and decode_fec=1 on a CELT packet (no in-band FEC: concealment, opus_decoder.c:655-657)."""
    cb = _cb()
    L = cb.lib()
    x = O.test_signal(48000, 2, 3, "tone")
    d, o, l, _ = O.encode_stream(x, 960, 64000)
    F = len(l)
    err = C.c_int(0)
    h = L.opus_decoder_create(48000, 2, C.byref(err))
    out = np.zeros((960, 2), dtype=np.int16)
    l2 = l.copy()
    l2[5] = 0
    l2[20:22] = 0
    rp, rr, rret = O.decode_stream(d, o, l2, 960, 2)
    for f in range(F):
        if l2[f] == 0:
            r = L.opus_decode(C.c_void_p(h), None, 0, O.ptr(out), 960, 0)
        else:
            pkt = d[o[f]:o[f] + l[f]].copy()
            r = L.opus_decode(C.c_void_p(h), O.ptr(pkt), int(l[f]), O.ptr(out), 960, 0)
        assert r == 960 and np.array_equal(out, rp[f * 960:(f + 1) * 960]), f
    L.opus_decoder_destroy(C.c_void_p(h))


_MULTICHUNK = r'''
import ctypes as C, sys, os
import numpy as np
sys.path.insert(0, os.path.join(os.getcwd(), "tests"))
import oracle_lib as O
import concentus_b200 as cb
import torch
L = cb.lib()
assert L.opus_b200_init(0) == 0
fs, ch, nsec = 960, 2, 4
kinds = ("music", "tone", "clicks", "noise")
datas, offs_all, lens_all, base = [], [], [], 0
n = 12
for s in range(n):
    x = O.test_signal(48000 * nsec, ch, 900 + s, kinds[s % 4])
    d, o, l, _ = O.encode_stream(x, fs, (64000, 96000, 160000)[s % 3], ch, vbr=1, cvbr=0)
    d, o = O.pack(d, o, l)
    l = l.copy()
    rs = np.random.RandomState(s)
    if s % 3 == 1:
        l[rs.rand(len(l)) < 0.15] = 0          # random loss: concealment state and the fold seed cross chunk boundaries
    if s % 3 == 2:
        for f in range(15, len(l), 37):
            l[f:f + 7] = 0                       # bursts past the noise-PLC threshold
    datas.append(d); offs_all.append(o + base); lens_all.append(l); base += len(d)
data = np.concatenate(datas); offs = np.stack(offs_all); lens = np.stack(lens_all)
F = lens.shape[1]
ref = [O.decode_stream(data, offs[s], lens[s], fs, ch) for s in range(n)]

def check(pcm, rets, fr, tag):
    pcm = pcm.reshape(n, F, -1); rets = rets.reshape(n, F)
    for s in range(n):
        rp, rr, rret = ref[s]
        assert np.array_equal(rret, rets[s]), (tag, "ret", s)
        bad = np.nonzero((rp.reshape(F, -1) != pcm[s]).any(axis=1))[0]
        assert bad.size == 0, (tag, "pcm", s, "first bad frame", int(bad[0]))
        assert int(rr[-1]) == int(fr[s]), (tag, "final range", s)

# host-buffer path, ONE call over all F packets: the library cuts it into chunks (CB200_IR_HOST_MB is tiny here)
dec = cb.DecoderBatch(n, 48000, ch)
p, r = dec.decode_span(data, offs.reshape(-1), lens.reshape(-1), F, fs)
check(p, r, dec.final_ranges(), "host")
dec.close()
# two host calls, the second one starting inside a loss run that covers more than its whole first chunk: the runs of its
# second chunk have nothing received to walk back to and take their context from the call-start snapshot while stage B of the
# first chunk is already advancing the live state (the race tools/parity_sweep.py found)
lens2 = lens.copy()
cut = 101
for s in range(n):
    lens2[s, cut - (s % 3):cut + 14 + 5 * (s % 4)] = 0
ref2 = [O.decode_stream(data, offs[s], lens2[s], fs, ch) for s in range(n)]
dec = cb.DecoderBatch(n, 48000, ch)
pa, ra = dec.decode_span(data, offs[:, :cut].reshape(-1), lens2[:, :cut].reshape(-1), cut, fs)
pb, rb = dec.decode_span(data, offs[:, cut:].reshape(-1), lens2[:, cut:].reshape(-1), F - cut, fs)
fr2 = dec.final_ranges()
dec.close()
p2 = np.concatenate([pa.reshape(n, cut, -1), pb.reshape(n, F - cut, -1)], axis=1)
r2 = np.concatenate([ra.reshape(n, cut), rb.reshape(n, F - cut)], axis=1)
ref_keep, ref = ref, ref2
check(p2, r2, fr2, "two calls, loss across the boundary")
ref = ref_keep
# device-resident path
dev = torch.device("cuda", 0)
d_blob = torch.from_numpy(data).to(dev); d_offs = torch.from_numpy(offs.reshape(-1).astype(np.int64)).to(dev)
d_lens = torch.from_numpy(lens.reshape(-1).astype(np.int32)).to(dev)
d_pcm = torch.zeros((n * F * fs * ch,), dtype=torch.int16, device=dev); d_ret = torch.zeros((n * F,), dtype=torch.int32, device=dev)
dec = cb.DecoderBatch(n, 48000, ch)
rc = L.opus_decode_span_device(dec.handles, n, F, C.c_void_p(d_blob.data_ptr()), C.c_void_p(d_offs.data_ptr()), C.c_void_p(d_lens.data_ptr()),
                               C.c_void_p(d_pcm.data_ptr()), fs, C.c_void_p(d_ret.data_ptr()))
assert rc == 0, rc
torch.cuda.synchronize(); L.opus_b200_synchronize()
check(d_pcm.cpu().numpy(), d_ret.cpu().numpy(), dec.final_ranges(), "device")
dec.close()
print("chunks-ok", F)
'''


def test_decode_multichunk_pipeline():
    """The time-chunked, double-buffered three-stage pipeline the bench runs on (DESIGN.md §3): forced here with a 2 MB IR budget
    so that 200 packets x 12 streams take ~14 chunks, with random and burst packet loss so that the fold seed, the loss streak
    and the concealment state all cross chunk boundaries.  Host-buffer and device-resident entry points, vs the oracle."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, CB200_IR_MB="2", CB200_IR_HOST_MB="2")
    out = subprocess.run([sys.executable, "-c", _MULTICHUNK], capture_output=True, text=True, cwd=root, env=env, timeout=600)
    assert out.returncode == 0 and "chunks-ok" in out.stdout, out.stdout[-2000:] + out.stderr[-4000:]


def test_rejected_packet_leaves_zero_pcm_and_untouched_state():
    """A packet the decoder rejects inside a span (a code-3 TOC with no count byte: OPUS_INVALID_PACKET, opus.c:228) must not
    touch the stream's state (the following packets decode as in the reference, which skips it the same way) and must not hand
    back stale buffer contents: its PCM row is zeros.  Found by tools/parity_sweep.py (wide mode)."""
    cb = _cb()
    ch, fs = 2, 960
    x = O.test_signal(48000, ch, 77, "music")
    d, o, l, _ = O.encode_stream(x, fs, 64000, ch, vbr=1, cvbr=0)
    d, o = O.pack(d, o, l)
    F = len(l)
    dec = cb.DecoderBatch(1, 48000, ch)
    dec.decode_span(d, o, l, F, fs)                 # fills the library's PCM staging with non-zero audio
    dec.close()
    d2 = d.copy()
    l2 = l.copy()
    for f in (7, 20):
        d2[o[f]] = 0xFF                              # CELT fullband stereo, code 3
        l2[f] = 1
    rp, rr, rret = O.decode_stream(d2, o, l2, fs, ch)
    assert rret[7] == -4 and rret[20] == -4
    dec = cb.DecoderBatch(1, 48000, ch)
    p, r = dec.decode_span(d2, o, l2, F, fs)
    fr = dec.final_ranges()
    dec.close()
    assert np.array_equal(r, rret)
    p = p.reshape(F, -1)
    assert not p[7].any() and not p[20].any()
    ok = np.ones(F, dtype=bool)
    ok[[7, 20]] = False
    assert np.array_equal(p[ok], rp.reshape(F, -1)[ok])
    assert int(fr[0]) == int(rr[-1])


def test_decoder_gain_ctl():
    """OPUS_SET_GAIN (src/opus_decoder.c:836-846, applied per sample in opus_decode_native :700-711; here inside stage C):
    positive and negative Q8 gains incl. ones that saturate, changed in the middle of the stream between two span calls, mono
    and stereo, 48 and 16 kHz output, with lost packets (the gain also scales concealed audio)."""
    cb = _cb()
    L = cb.lib()
    G = np.load(DECODER_CTL)
    cases = [(2, 960, 48000, 768, -1500), (1, 480, 48000, -3000, 2500), (2, 960, 16000, 5000, 300), (2, 240, 48000, 32767, -32768)]
    for k, (ch, fs, dFs, g1, g2) in enumerate(cases):
        x = O.test_signal(48000, ch, 50 + k, ("music", "noise", "tone", "clicks")[k])
        d, o, l, _ = O.encode_stream(x, fs, 64000, ch, vbr=1, cvbr=0)
        d, o = O.pack(d, o, l)
        l = l.copy()
        l[11::13] = 0
        F = len(l)
        cut = F // 2
        dfs = fs * dFs // 48000
        rret, rcrc = G["gain%d_rets" % k], G["gain%d_pcm_crc" % k]
        dec = cb.DecoderBatch(1, dFs, ch)
        h = C.c_void_p(dec.handles[0])
        assert L.opus_decoder_ctl(h, cb.OPUS_SET_GAIN_REQUEST, C.c_int32(g1)) == 0
        p1, r1 = dec.decode_span(d, o[:cut], l[:cut], cut, dfs)
        assert L.opus_decoder_ctl(h, cb.OPUS_SET_GAIN_REQUEST, C.c_int32(g2)) == 0
        got = C.c_int32(0)
        assert L.opus_decoder_ctl(h, 4045, C.byref(got)) == 0 and got.value == g2      # OPUS_GET_GAIN
        p2, r2 = dec.decode_span(d, o[cut:], l[cut:], F - cut, dfs)
        dec.close()
        assert np.array_equal(np.concatenate([r1, r2]), rret), (ch, fs, dFs)
        got_pcm = np.concatenate([p1, p2]).reshape(F, -1)
        bad = np.nonzero(_row_crc(got_pcm) != rcrc)[0]
        assert bad.size == 0, (ch, fs, dFs, g1, g2, "first bad frame", int(bad[0]))
    # out-of-range gains are rejected like the reference (opus_decoder.c:839)
    dec = cb.DecoderBatch(1, 48000, 2)
    assert L.opus_decoder_ctl(C.c_void_p(dec.handles[0]), cb.OPUS_SET_GAIN_REQUEST, C.c_int32(40000)) == -1
    dec.close()


def test_decoder_getters_and_reset_per_packet():
    """opus_decoder_ctl getters after every packet of the scalar API — OPUS_GET_PITCH (celt_decoder.c:1208, the post-filter
    period), OPUS_GET_LAST_PACKET_DURATION, OPUS_GET_BANDWIDTH, OPUS_GET_SAMPLE_RATE, OPUS_GET_FINAL_RANGE — and
    OPUS_RESET_STATE in the middle of a stream (src/opus_decoder.c:812-822), with lost packets; vs the reference."""
    cb = _cb()
    L = cb.lib()
    G = np.load(DECODER_CTL)
    for k, (ch, fs, dFs, kind, br) in enumerate(((2, 960, 48000, "tone", 64000), (1, 480, 24000, "music", 48000), (2, 240, 48000, "clicks", 128000))):
        x = O.test_signal(48000, ch, 90 + k, kind)
        d, o, l, _ = O.encode_stream(x, fs, br, ch, vbr=1, cvbr=0)
        d, o = O.pack(d, o, l)
        l = l.copy()
        l[6::11] = 0
        F = min(len(l), 60)
        reset_at = 23
        dfs = fs * dFs // 48000
        rret, rr, info, rcrc = (G["info%d_%s" % (k, n)] for n in ("rets", "ranges", "info", "pcm_crc"))
        err = C.c_int(0)
        L.opus_decoder_create.restype = C.c_void_p
        h = C.c_void_p(L.opus_decoder_create(dFs, ch, C.byref(err)))
        out = np.zeros((dfs, ch), dtype=np.int16)
        v = C.c_int32(0)
        u = C.c_uint32(0)
        for f in range(F):
            if f == reset_at:
                assert L.opus_decoder_ctl(h, cb.OPUS_RESET_STATE) == 0
            p = O.ptr(d[o[f]:]) if l[f] > 0 else None
            n = L.opus_decode(h, p, int(l[f]), O.ptr(out), dfs, 0)
            assert n == rret[f], (k, f, n, int(rret[f]))
            assert _row_crc([out[:max(n, 0)]])[0] == rcrc[f], (k, f)
            L.opus_decoder_ctl(h, cb.OPUS_GET_FINAL_RANGE_REQUEST, C.byref(u))
            assert u.value == int(rr[f]), (k, f, "final range")
            for j, req in enumerate((cb.OPUS_GET_PITCH_REQUEST, cb.OPUS_GET_LAST_PACKET_DURATION_REQUEST, cb.OPUS_GET_BANDWIDTH_REQUEST,
                                     cb.OPUS_GET_SAMPLE_RATE_REQUEST)):
                assert L.opus_decoder_ctl(h, req, C.byref(v)) == 0
                assert v.value == int(info[f, j]), (k, f, ("pitch", "last_packet_duration", "bandwidth", "sample_rate")[j], v.value, int(info[f, j]))
        L.opus_decoder_destroy(h)


def test_plc_packets_with_non_celt_toc_and_oversized_capacity():
    """(1) When max_data_bytes leaves no room for a frame the encoder emits "PLC frames": a TOC-only packet whose TOC says SILK
    for 40 / 60 ms frames (opus_encoder.c:1240-1270), CBR-padded to a code-3 packet with an empty frame.  The decoder conceals
    them from the CELT state, 40 / 60 ms in 20 ms pieces (opus_decoder.c:246-268) — not OPUS_UNIMPLEMENTED.  (2) A PCM
    capacity larger than the packet's duration: received packets return their own duration (the rest of the row reads zero),
    lost packets are concealed over the whole capacity.  Found by tools/parity_sweep.py (wide mode)."""
    cb = _cb()
    for k, (Fs, ch, ms, vbr, maxb, capmul) in enumerate(((48000, 2, 60, 0, 3, 1), (12000, 2, 60, 1, 3, 1), (16000, 1, 40, 0, 8, 1),
                                                         (48000, 2, 20, 1, 1276, 3), (48000, 1, 10, 1, 1276, 2), (24000, 2, 5, 0, 1276, 3))):
        fs = Fs * ms // 1000
        x = O.test_signal(Fs * 2, ch, 30 + k, ("music", "tone", "clicks")[k % 3])
        F = x.shape[0] // fs
        normal = O.encode_stream(x, fs, 64000, ch, Fs=Fs, vbr=vbr, cvbr=0, complexity=5, max_bytes=1276)
        tiny = O.encode_stream(x, fs, 64000, ch, Fs=Fs, vbr=vbr, cvbr=0, complexity=5, max_bytes=maxb)
        # a stream that alternates between real packets and what the starved encoder produced for the same frames
        data = np.concatenate([normal[0], tiny[0]])
        use_tiny = (np.arange(F) % 5) >= 3
        offs = np.where(use_tiny, tiny[1] + len(normal[0]), normal[1])
        lens = np.where(use_tiny, tiny[2], normal[2]).astype(np.int32)
        lens[7::11] = 0
        cap = fs * capmul
        rp, rr, rret = O.decode_stream(data, offs, lens, cap, ch, Fs=Fs)
        assert (rret > 0).all(), (k, rret[:12])
        dec = cb.DecoderBatch(1, Fs, ch)
        p1, r1 = dec.decode_span(data, offs[:F // 2], lens[:F // 2], F // 2, cap)
        p2, r2 = dec.decode_span(data, offs[F // 2:], lens[F // 2:], F - F // 2, cap)
        fr = dec.final_ranges()
        dec.close()
        assert np.array_equal(np.concatenate([r1, r2]), rret), (k, Fs, ms, maxb)
        got = np.concatenate([p1, p2]).reshape(F, -1)
        bad = np.nonzero((rp.reshape(F, -1) != got).any(axis=1))[0]
        assert bad.size == 0, (k, Fs, ms, maxb, capmul, "first bad row", int(bad[0]))
        assert int(fr[0]) == int(rr[-1])

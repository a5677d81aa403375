"""Multistream decoder on the GPU (opus_multistream_decode, _span, _span_device).  The reference multistream decoder is per-stream
opus_decode_native plus a channel copy, so it is pinned two ways: against the reference's results for the streams of the golden
fixtures (tests/golden/*.npz: return codes, final ranges and CRC-32 of the PCM per packet), and against fresh single-stream decoders
of this library — which the rest of the suite pins to the reference — on the same packets.  Multistream packets are framed here
in plain Python (tests/ms_framing.py)."""
import ctypes as C
import os
import subprocess
import sys
import zlib

import numpy as np
import pytest

import ms_framing as M
import oracle_lib as O

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
OK, BAD_ARG, BUFFER_TOO_SMALL, INVALID_PACKET, UNIMPLEMENTED = 0, -1, -2, -4, -5


def _cb():
    import concentus_b200 as cb
    assert cb.lib().opus_b200_init(0) == 0, "CUDA device required: no CPU fallback exists"
    return cb


def _crc(rows):
    return np.array([zlib.crc32(np.ascontiguousarray(r).tobytes()) for r in rows], dtype=np.uint32)


def _stream_state(L, h, s):
    p = C.c_void_p(0)
    assert L.opus_multistream_decoder_ctl(C.c_void_p(h), 5122, C.c_int32(s), C.byref(p)) == OK
    return p


def _ranges(L, h, S):
    """(final range of every stream through OPUS_MULTISTREAM_GET_DECODER_STATE, multistream OPUS_GET_FINAL_RANGE)."""
    v = C.c_uint32(0)
    out = []
    for s in range(S):
        assert L.opus_decoder_ctl(_stream_state(L, h, s), 4031, C.byref(v)) == OK
        out.append(v.value)
    assert L.opus_multistream_decoder_ctl(C.c_void_p(h), 4031, C.byref(v)) == OK
    return out, v.value


def _stream_channels(mapping, S, coupled):
    """Output columns that carry each stream: coupled s -> (col of 2s, col of 2s+1), mono s -> (col of coupled+s,)."""
    mapping = list(mapping)
    cols = []
    for s in range(S):
        ks = (2 * s, 2 * s + 1) if s < coupled else (coupled + s,)
        cols.append(tuple(mapping.index(k) for k in ks))
    return cols


def _compose(stream_pcm, mapping, S, coupled, rows):
    """Single-stream PCM [S][rows, ch] -> multistream PCM [rows, channels] (the reference's channel copy)."""
    out = np.zeros((rows, len(mapping)), dtype=np.int16)
    for c, k in enumerate(mapping):
        if k == 255:
            continue
        if k < 2 * coupled:
            out[:, c] = stream_pcm[k // 2][:, k & 1]
        else:
            out[:, c] = stream_pcm[k - coupled][:, 0]
    return out


# ---------------------------------------------------------------------------------------------------------------------------
# 1. the reference's results for the golden streams
# ---------------------------------------------------------------------------------------------------------------------------
GOLDEN_LAYOUTS = [
    # (fixtures of the coupled streams, then the mono ones), coupled, mapping
    (["music_st_20ms_128k_vbr", "music_st_20ms_64k_cbr", "music_mono_20ms_32k_vbr"], 2, [0, 1, 2, 3, 4]),
    (["music_st_20ms_128k_vbr", "music_st_20ms_64k_cbr", "music_mono_20ms_32k_vbr"], 2, [0, 1, 255, 2, 3, 4, 1]),
    (["noise_st_2p5ms_510k_cbr", "tone_st_2p5ms_32k_vbr_monocoded"], 2, [0, 1, 2, 3]),
    (["clicks_mono_5ms_48k_vbr"], 0, [0]),
    (["clicks_mono_5ms_48k_vbr"], 0, [0, 0]),
    (["tone_st_10ms_96k_cvbr"], 1, [0, 1]),
]


@pytest.mark.parametrize("names,coupled,mapping", GOLDEN_LAYOUTS)
def test_multistream_matches_reference_results_of_golden_streams(names, coupled, mapping):
    cb = _cb()
    L = cb.lib()
    G = [np.load(os.path.join(GOLDEN, n + ".npz")) for n in names]
    S, ch = len(names), len(mapping)
    fs = int(G[0]["frame_size"])
    F = len(G[0]["lens"])
    assert all(int(g["frame_size"]) == fs and len(g["lens"]) == F for g in G)
    assert [int(g["channels"]) for g in G] == [2] * coupled + [1] * (S - coupled)
    pkts = [M.ms_packet([bytes(g["data"][g["offs"][f]:g["offs"][f] + g["lens"][f]]) for g in G]) for f in range(F)]
    blob, offs, lens = M.ms_blob(pkts)
    cols = _stream_channels(mapping, S, coupled)

    def check(pcm, rets, tag):
        pcm = pcm.reshape(F, fs, ch)
        for s, g in enumerate(G):
            assert np.array_equal(rets, g["rets"]), (tag, names[s], "ret")
            assert np.array_equal(_crc(pcm[:, :, list(cols[s])]), g["pcm_crc"]), (tag, names[s], "pcm")
        for c, k in enumerate(mapping):
            if k == 255:
                assert not pcm[:, :, c].any(), (tag, "silent channel")
            else:
                assert np.array_equal(pcm[:, :, c], pcm[:, :, mapping.index(k)]), (tag, "duplicated channel")

    def check_ranges(h, f, tag):
        per, x = _ranges(L, h, S)
        assert per == [int(g["dec_ranges"][f]) for g in G], (tag, f)
        assert x == int(np.bitwise_xor.reduce(np.array(per, dtype=np.uint32))), (tag, f)

    err = C.c_int(0)
    mp = np.array(mapping, dtype=np.uint8)
    # scalar calls, ranges after every packet
    h = L.opus_multistream_decoder_create(48000, ch, S, coupled, O.ptr(mp), C.byref(err))
    assert h and err.value == 0
    pcm = np.zeros((F, fs, ch), dtype=np.int16)
    rets = np.zeros(F, dtype=np.int32)
    for f in range(F):
        p = np.frombuffer(pkts[f], dtype=np.uint8).copy()
        rets[f] = L.opus_multistream_decode(C.c_void_p(h), O.ptr(p), len(p), O.ptr(pcm[f]), fs, 0)
        check_ranges(h, f, "scalar")
    check(pcm, rets, "scalar")
    L.opus_multistream_decoder_destroy(C.c_void_p(h))
    # host spans, two calls
    dec = cb.MSDecoderBatch(1, 48000, ch, S, coupled, mapping)
    F1 = F // 2 + 1
    p1, r1 = dec.decode_span(blob, offs[:F1], lens[:F1], F1, fs)
    p2, r2 = dec.decode_span(blob, offs[F1:], lens[F1:], F - F1, fs)
    check(np.concatenate([p1, p2]), np.concatenate([r1, r2]), "host span")
    check_ranges(dec.handles[0], F - 1, "host span")
    dec.close()
    # device spans, two calls
    import torch
    dev = torch.device("cuda", 0)
    dec = cb.MSDecoderBatch(1, 48000, ch, S, coupled, mapping)
    d_blob = torch.from_numpy(blob).to(dev)
    outs, rs = [], []
    for a, b in ((0, F1), (F1, F)):
        d_offs = torch.from_numpy(offs[a:b].copy()).to(dev)
        d_lens = torch.from_numpy(lens[a:b].copy()).to(dev)
        d_pcm = torch.full(((b - a) * fs * ch,), 77, dtype=torch.int16, device=dev)
        d_ret = torch.zeros((b - a,), dtype=torch.int32, device=dev)
        rc = L.opus_multistream_decode_span_device(dec.handles, 1, b - a, C.c_void_p(d_blob.data_ptr()), C.c_void_p(d_offs.data_ptr()),
                                                   C.c_void_p(d_lens.data_ptr()), C.c_void_p(d_pcm.data_ptr()), fs,
                                                   C.c_void_p(d_ret.data_ptr()))
        assert rc == OK
        assert L.opus_b200_synchronize() == OK
        outs.append(d_pcm.cpu().numpy())
        rs.append(d_ret.cpu().numpy())
    check(np.concatenate(outs), np.concatenate(rs), "device span")
    check_ranges(dec.handles[0], F - 1, "device span")
    dec.close()


# ---------------------------------------------------------------------------------------------------------------------------
# 2. composition at scale: the same packets through fresh single-stream decoders
# ---------------------------------------------------------------------------------------------------------------------------
def _make_layout_streams(rs, n, S, coupled, F10):
    """Per decoder m and stream s: F10 ordinary 10 ms packets (uint8 blob, offs, lens) of a random signal / bitrate / VBR mode."""
    out = []
    for m in range(n):
        row = []
        for s in range(S):
            ch = 2 if s < coupled else 1
            kind = ("music", "tone", "noise", "clicks")[rs.randint(4)]
            pcm = O.test_signal(480 * F10, ch, int(rs.randint(1, 1 << 30)), kind)
            br = int(rs.choice([16000, 32000, 64000, 96000, 160000])) * ch
            vbr = int(rs.randint(2))
            d, o, l, _ = O.encode_stream(pcm, 480, br, ch, vbr=vbr, cvbr=int(rs.randint(2)) if vbr else 0, pin=False)
            row.append([bytes(d[o[f]:o[f] + l[f]]) for f in range(F10)])
        out.append(row)
    return out


def _group_packets(rs, ten_ms, groups, pad_prob=0.15):
    """Merge consecutive 10 ms packets of one stream into one packet per group size (1, 2, 4 or 6 frames: 10..60 ms)."""
    out, f = [], 0
    for gsz in groups:
        frames = [M.parse(p)[2][0] for p in ten_ms[f:f + gsz]]
        toc = ten_ms[f][0] & 0xFC
        f += gsz
        if gsz == 1:
            pkt = ten_ms[f - 1]
        elif gsz == 2 and len(frames[0]) == len(frames[1]):
            pkt = M.build(toc, 1, frames)
        elif gsz == 2:
            pkt = M.build(toc, 2, frames)
        else:
            pkt = M.build(toc, 3, frames)
        if rs.rand() < pad_prob:
            pkt = M.pad_packet(pkt, int(rs.choice([1, 3, 200, 600])))
        out.append(pkt)
    return out


def _composition_case(seed, n=3, F10=48, host=True, device=True, scalar=False):
    """One random layout: n multistream decoders (different mappings) vs n*S single-stream decoders on the same packets."""
    cb = _cb()
    L = cb.lib()
    rs = np.random.RandomState(seed)
    S = int(rs.randint(1, 9))
    coupled = int(rs.randint(0, S + 1))
    ch = int(rs.randint(1, 17))
    nk = S + coupled
    maps = []
    for m in range(n):
        mp = [int(x) for x in rs.randint(0, nk, size=ch)]
        for c in range(ch):
            if rs.rand() < 0.12:
                mp[c] = 255
        maps.append(mp)
    ten = _make_layout_streams(rs, n, S, coupled, F10)
    groups = []
    left = F10
    while left > 0:
        g = int(rs.choice([1, 2, 4, 6]))
        g = min(g, left)
        if g == 3 or g == 5:
            g = 1
        groups.append(g)
        left -= g
    F = len(groups)
    lost = rs.rand(n, F) < 0.08
    frame_size = 2880
    subs = [[_group_packets(rs, ten[m][s], groups) for s in range(S)] for m in range(n)]
    ms = []
    for m in range(n):
        for f in range(F):
            ms.append(b"" if lost[m, f] else M.ms_packet([subs[m][s][f] for s in range(S)]))
    blob, offs, lens = M.ms_blob(ms)
    # reference: single-stream spans of the undelimited sub-packets (lost = len 0), one call per channel count
    ref_pcm = [[None] * S for _ in range(n)]
    ref_ret = np.zeros((n, S, F), dtype=np.int32)
    ref_rng = np.zeros((n, S), dtype=np.uint32)
    for chn, streams in ((2, range(coupled)), (1, range(coupled, S))):
        ids = [(m, s) for m in range(n) for s in streams]
        if not ids:
            continue
        pk = [b"" if lost[m, f] else subs[m][s][f] for (m, s) in ids for f in range(F)]
        b, o, l = M.ms_blob(pk)
        dec = cb.DecoderBatch(len(ids), 48000, chn)
        p, r = dec.decode_span(b, o, l, F, frame_size)
        fr = dec.final_ranges()
        dec.close()
        p = p.reshape(len(ids), F, frame_size, chn)
        r = r.reshape(len(ids), F)
        for i, (m, s) in enumerate(ids):
            ref_pcm[m][s] = p[i]
            ref_ret[m, s] = r[i]
            ref_rng[m, s] = fr[i]
    assert (ref_ret > 0).all(), "inputs are meant to decode"
    want = np.zeros((n, F, frame_size, ch), dtype=np.int16)
    for m in range(n):
        for f in range(F):
            want[m, f] = _compose([ref_pcm[m][s][f] for s in range(S)], maps[m], S, coupled, frame_size)
    want_ret = ref_ret[:, 0, :]
    assert (ref_ret == want_ret[:, None, :]).all()

    def check(pcm, rets, dec, tag):
        pcm = pcm.reshape(n, F, frame_size, ch)
        assert np.array_equal(rets.reshape(n, F), want_ret), (tag, seed)
        bad = np.argwhere((pcm != want).any(axis=(2, 3)))
        assert bad.size == 0, (tag, seed, "first bad (decoder, packet)", bad[0].tolist())
        for m in range(n):
            per, x = _ranges(L, dec.handles[m], S)
            assert per == ref_rng[m].tolist(), (tag, seed, m)
            assert x == int(np.bitwise_xor.reduce(ref_rng[m])), (tag, seed, m)
    if host:
        dec = cb.MSDecoderBatch(n, 48000, ch, S, coupled, maps)
        idx = np.arange(n * F).reshape(n, F)
        cut = F // 3
        pa, ra = dec.decode_span(blob, offs[idx[:, :cut].reshape(-1)], lens[idx[:, :cut].reshape(-1)], cut, frame_size)
        pb, rb = dec.decode_span(blob, offs[idx[:, cut:].reshape(-1)], lens[idx[:, cut:].reshape(-1)], F - cut, frame_size)
        pcm = np.concatenate([pa.reshape(n, cut, -1), pb.reshape(n, F - cut, -1)], axis=1)
        rets = np.concatenate([ra.reshape(n, cut), rb.reshape(n, F - cut)], axis=1)
        check(pcm, rets, dec, "host span")
        dec.close()
    if device:
        import torch
        dev = torch.device("cuda", 0)
        dec = cb.MSDecoderBatch(n, 48000, ch, S, coupled, maps)
        d_blob = torch.from_numpy(blob).to(dev)
        d_offs = torch.from_numpy(offs).to(dev)
        d_lens = torch.from_numpy(lens).to(dev)
        d_pcm = torch.full((n * F * frame_size * ch,), -5, dtype=torch.int16, device=dev)
        d_ret = torch.zeros((n * F,), dtype=torch.int32, device=dev)
        rc = L.opus_multistream_decode_span_device(dec.handles, n, F, C.c_void_p(d_blob.data_ptr()), C.c_void_p(d_offs.data_ptr()),
                                                   C.c_void_p(d_lens.data_ptr()), C.c_void_p(d_pcm.data_ptr()), frame_size,
                                                   C.c_void_p(d_ret.data_ptr()))
        assert rc == OK
        assert L.opus_b200_synchronize() == OK
        check(d_pcm.cpu().numpy(), d_ret.cpu().numpy(), dec, "device span")
        dec.close()
    if scalar:
        dec = cb.MSDecoderBatch(n, 48000, ch, S, coupled, maps)
        pcm = np.zeros((n, F, frame_size, ch), dtype=np.int16)
        rets = np.zeros((n, F), dtype=np.int32)
        for m in range(n):
            for f in range(F):
                p = np.frombuffer(ms[m * F + f] + b"\0", dtype=np.uint8).copy()
                rets[m, f] = L.opus_multistream_decode(C.c_void_p(dec.handles[m]), O.ptr(p), len(ms[m * F + f]), O.ptr(pcm[m, f]),
                                                       frame_size, 0)
        check(pcm, rets, dec, "scalar")
        dec.close()
    return S, coupled, ch


@pytest.mark.parametrize("seed", [1, 2, 3, 4, 5, 6])
def test_multistream_composition_random_layouts(seed):
    _composition_case(seed, scalar=seed == 1)


_MULTICHUNK = r'''
import sys
sys.path.insert(0, "tests")
import test_multistream_gpu as T
for seed in (11, 12):
    T._composition_case(seed, n=4, F10=160)
print("ms-chunks-ok")
'''


def test_multistream_multichunk_pipeline():
    """The time-chunked pipeline (a 2 MB IR budget: many chunks per call) with the elementary staging double-buffered between the
    decoder stages and the gather."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, CB200_IR_MB="2", CB200_IR_HOST_MB="2")
    out = subprocess.run([sys.executable, "-c", _MULTICHUNK], capture_output=True, text=True, cwd=root, env=env, timeout=900)
    assert out.returncode == 0 and "ms-chunks-ok" in out.stdout, out.stdout[-2000:] + out.stderr[-4000:]


# ---------------------------------------------------------------------------------------------------------------------------
# 3. rejections leave every stream untouched
# ---------------------------------------------------------------------------------------------------------------------------
def _golden_subpackets():
    G = [np.load(os.path.join(GOLDEN, n + ".npz")) for n in ("music_st_20ms_128k_vbr", "music_st_20ms_64k_cbr", "music_mono_20ms_32k_vbr")]
    F = len(G[0]["lens"])
    return [[bytes(g["data"][g["offs"][f]:g["offs"][f] + g["lens"][f]]) for g in G] for f in range(F)], F


def _rejects(good_next):
    """Rejected multistream packets of 3 streams (2 coupled, 1 mono) and the code each must give (frame_size 960)."""
    a, b, c = good_next
    silk = M.build(0x48, 0, [bytes(range(1, 30))])
    forty = M.build(a[0] & 0xFC, 3, [M.parse(a)[2][0]] * 2)   # 40 ms
    ms = bytearray(M.ms_packet([a, b, c]))
    garbled = bytearray(ms)
    garbled[1], garbled[2] = 255, 255
    return [
        (M.ms_packet([a, forty, c]), INVALID_PACKET),        # durations differ
        (bytes(ms[:4]), INVALID_PACKET),                      # len < 2S-1
        (bytes(ms[:len(M.self_delimit(a)) - 3]), INVALID_PACKET),   # truncated inside stream 0
        (bytes(garbled), INVALID_PACKET),                     # garbled self-delimited length
        (M.ms_packet([a, silk, c]), UNIMPLEMENTED),           # SILK frame in stream 1
        (M.ms_packet([forty, forty, forty]), BUFFER_TOO_SMALL),   # 40 ms in 960 samples
    ]


def test_multistream_rejections_leave_every_stream_untouched():
    cb = _cb()
    L = cb.lib()
    subs, F = _golden_subpackets()
    mapping = [0, 1, 2, 3, 4]
    fs = 960
    good = [M.ms_packet(p) for p in subs]
    # decoder 0 gets rejected packets in between, decoder 1 (its neighbour in the span) only good ones
    seq0, expect0 = [], []
    for f in range(F):
        if f in (3, 10, 17, 24, 31, 38):
            for pkt, code in _rejects(subs[f]):
                seq0.append(pkt)
                expect0.append(code)
        seq0.append(good[f])
        expect0.append(None)
    seq1 = [good[(f * 7) % F] for f in range(len(seq0))]
    blob, offs, lens = M.ms_blob(seq0 + seq1)
    Fx = len(seq0)
    dec = cb.MSDecoderBatch(2, 48000, 5, 3, 2, mapping)
    pcm, rets = dec.decode_span(blob, offs, lens, Fx, fs)
    pcm = pcm.reshape(2, Fx, fs, 5)
    rets = rets.reshape(2, Fx)
    # what fresh decoders give without the rejected packets (decoder 0 has fewer: one span per decoder)
    keep = [i for i in range(Fx) if expect0[i] is None]
    b2, o2, l2 = M.ms_blob([seq0[i] for i in keep] + seq1)
    r0 = cb.MSDecoderBatch(1, 48000, 5, 3, 2, mapping)
    p0, q0 = r0.decode_span(b2, o2[:len(keep)], l2[:len(keep)], len(keep), fs)
    r1 = cb.MSDecoderBatch(1, 48000, 5, 3, 2, mapping)
    p1, q1 = r1.decode_span(b2, o2[len(keep):], l2[len(keep):], Fx, fs)
    p0 = p0.reshape(len(keep), fs, 5)
    for i in range(Fx):
        if expect0[i] is not None:
            assert rets[0, i] == expect0[i], (i, rets[0, i], expect0[i])
            assert not pcm[0, i].any()
    assert np.array_equal(rets[0, keep], q0)
    assert np.array_equal(pcm[0, keep], p0)
    assert np.array_equal(rets[1], q1) and np.array_equal(pcm[1].reshape(-1, 5), p1)
    for s in range(3):
        v0, v1 = C.c_uint32(0), C.c_uint32(0)
        L.opus_decoder_ctl(_stream_state(L, dec.handles[0], s), 4031, C.byref(v0))
        L.opus_decoder_ctl(_stream_state(L, r0.handles[0], s), 4031, C.byref(v1))
        assert v0.value == v1.value
    # the scalar call: same codes, the next packet decodes as if the rejected one had not been sent
    err = C.c_int(0)
    mp = np.array(mapping, dtype=np.uint8)
    h = L.opus_multistream_decoder_create(48000, 5, 3, 2, O.ptr(mp), C.byref(err))
    out = np.zeros((fs, 5), dtype=np.int16)
    k = 0
    for i in range(Fx):
        p = np.frombuffer(seq0[i] + b"\0", dtype=np.uint8).copy()
        r = L.opus_multistream_decode(C.c_void_p(h), O.ptr(p), len(seq0[i]), O.ptr(out), fs, 0)
        if expect0[i] is not None:
            assert r == expect0[i], (i, r)
        else:
            assert r == fs and np.array_equal(out, p0[k]), i
            k += 1
    # too small a frame_size for the scalar call is BUFFER_TOO_SMALL too, and leaves the state as it was
    p = np.frombuffer(good[0], dtype=np.uint8).copy()
    assert L.opus_multistream_decode(C.c_void_p(h), O.ptr(p), len(good[0]), O.ptr(out), 480, 0) == BUFFER_TOO_SMALL
    L.opus_multistream_decoder_destroy(C.c_void_p(h))
    for d in (dec, r0, r1):
        d.close()


# ---------------------------------------------------------------------------------------------------------------------------
# 4. state: memcpy, reset, gain, getters, sync
# ---------------------------------------------------------------------------------------------------------------------------
def _single_refs(cb, subs, F, fs, lost=(), gain=0, reset_at=None):
    """Single-stream decoders (2 coupled + 1 mono) over the golden sub-packets: ([S] pcm [F, fs, ch], rets, getters per packet)."""
    L = cb.lib()
    out = []
    for s, chn in enumerate((2, 2, 1)):
        dec = cb.DecoderBatch(1, 48000, chn)
        h = C.c_void_p(dec.handles[0])
        if gain:
            assert L.opus_decoder_ctl(h, cb.OPUS_SET_GAIN_REQUEST, C.c_int32(gain)) == OK
        pcm = np.zeros((F, fs, chn), dtype=np.int16)
        info = np.zeros((F, 3), dtype=np.int64)
        v = C.c_int32(0)
        for f in range(F):
            if f == reset_at:
                assert L.opus_decoder_ctl(h, cb.OPUS_RESET_STATE) == OK
            pkt = b"" if f in lost else subs[f][s]
            p = np.frombuffer(pkt + b"\0", dtype=np.uint8).copy()
            assert L.opus_decode(h, O.ptr(p), len(pkt), O.ptr(pcm[f]), fs, 0) == fs
            for j, req in enumerate((cb.OPUS_GET_BANDWIDTH_REQUEST, cb.OPUS_GET_LAST_PACKET_DURATION_REQUEST, 4031)):
                L.opus_decoder_ctl(h, req, C.byref(v))
                info[f, j] = v.value & 0xFFFFFFFF
        out.append((pcm, info))
        dec.close()
    return out


def test_multistream_state_memcpy_reset_gain_getters():
    cb = _cb()
    L = cb.lib()
    subs, F = _golden_subpackets()
    fs = 960
    mapping = [4, 0, 1, 2, 3]
    mp = np.array(mapping, dtype=np.uint8)
    good = [M.ms_packet(p) for p in subs]
    lost = {7, 8, 30}
    pk = [b"" if f in lost else good[f] for f in range(F)]
    blob, offs, lens = M.ms_blob(pk)
    size = L.opus_multistream_decoder_get_size(3, 2)
    err = C.c_int(0)

    def want(refs, f):
        return _compose([refs[s][0][f] for s in range(3)], mapping, 3, 2, fs)

    # memcpy of a live (device-resident) decoder between spans: the clone takes the state over, and the original goes on
    # identically after it
    refs = _single_refs(cb, subs, F, fs, lost=lost)
    dec = cb.MSDecoderBatch(1, 48000, 5, 3, 2, mapping)
    cut = 20
    p1, r1 = dec.decode_span(blob, offs[:cut], lens[:cut], cut, fs)
    clone = C.create_string_buffer(size)
    C.memmove(clone, dec.handles[0], size)
    hc = C.cast(clone, C.c_void_p).value
    p3 = np.zeros((F - cut, fs, 5), dtype=np.int16)
    r3 = np.zeros(F - cut, dtype=np.int32)
    hh = (C.c_void_p * 1)(hc)
    assert L.opus_multistream_decode_span(hh, 1, F - cut, O.ptr(blob), O.ptr(offs[cut:].copy()), O.ptr(lens[cut:].copy()), O.ptr(p3), fs,
                                          O.ptr(r3)) == OK
    p2, r2 = dec.decode_span(blob, offs[cut:], lens[cut:], F - cut, fs)
    allp = np.concatenate([p1, p2]).reshape(F, fs, 5)
    assert (np.concatenate([r1, r2]) == fs).all() and (r3 == fs).all()
    for f in range(F):
        assert np.array_equal(allp[f], want(refs, f)), f
        if f >= cut:
            assert np.array_equal(p3[f - cut], want(refs, f)), f
    assert _ranges(L, hc, 3)[0] == [int(refs[s][1][-1, 2]) for s in range(3)]
    assert L.opus_multistream_decoder_sync(hh, 1) == OK
    assert L.opus_multistream_decoder_sync(dec.handles, 1) == OK
    dec.close()
    # OPUS_RESET_STATE mid-stream, OPUS_SET_GAIN, getters after every packet (scalar calls) and after spans + sync
    for gain in (0, -2500, 1800):
        refs = _single_refs(cb, subs, F, fs, lost=lost, gain=gain, reset_at=25)
        h = L.opus_multistream_decoder_create(48000, 5, 3, 2, O.ptr(mp), C.byref(err))
        assert h and err.value == 0
        hv = C.c_void_p(h)
        if gain:
            assert L.opus_multistream_decoder_ctl(hv, cb.OPUS_SET_GAIN_REQUEST, C.c_int32(gain)) == OK
        out = np.zeros((fs, 5), dtype=np.int16)
        v = C.c_int32(0)
        for f in range(F):
            if f == 25:
                assert L.opus_multistream_decoder_ctl(hv, cb.OPUS_RESET_STATE) == OK
            p = np.frombuffer(pk[f] + b"\0", dtype=np.uint8).copy()
            assert L.opus_multistream_decode(hv, O.ptr(p), len(pk[f]), O.ptr(out), fs, 0) == fs
            assert np.array_equal(out, want(refs, f)), (gain, f)
            assert L.opus_multistream_decoder_ctl(hv, cb.OPUS_GET_BANDWIDTH_REQUEST, C.byref(v)) == OK and v.value == refs[0][1][f, 0]
            assert L.opus_multistream_decoder_ctl(hv, cb.OPUS_GET_LAST_PACKET_DURATION_REQUEST, C.byref(v)) == OK and v.value == refs[0][1][f, 1]
            assert L.opus_multistream_decoder_ctl(hv, cb.OPUS_GET_GAIN_REQUEST, C.byref(v)) == OK and v.value == gain
            assert L.opus_multistream_decoder_ctl(hv, cb.OPUS_GET_SAMPLE_RATE_REQUEST, C.byref(v)) == OK and v.value == 48000
            assert _ranges(L, h, 3)[0] == [int(refs[s][1][f, 2]) for s in range(3)], (gain, f)
        L.opus_multistream_decoder_destroy(hv)
        # the same through two spans with the reset and the gain between them
        dec = cb.MSDecoderBatch(1, 48000, 5, 3, 2, mapping)
        hv = C.c_void_p(dec.handles[0])
        if gain:
            assert L.opus_multistream_decoder_ctl(hv, cb.OPUS_SET_GAIN_REQUEST, C.c_int32(gain)) == OK
        pa, _ = dec.decode_span(blob, offs[:25], lens[:25], 25, fs)
        assert L.opus_multistream_decoder_ctl(hv, cb.OPUS_RESET_STATE) == OK
        pb, _ = dec.decode_span(blob, offs[25:], lens[25:], F - 25, fs)
        allp = np.concatenate([pa, pb]).reshape(F, fs, 5)
        for f in range(F):
            assert np.array_equal(allp[f], want(refs, f)), ("span", gain, f)
        assert L.opus_multistream_decoder_sync(dec.handles, 1) == OK
        assert L.opus_multistream_decoder_ctl(hv, cb.OPUS_GET_LAST_PACKET_DURATION_REQUEST, C.byref(v)) == OK and v.value == fs
        assert _ranges(L, dec.handles[0], 3)[0] == [int(refs[s][1][-1, 2]) for s in range(3)]
        dec.close()

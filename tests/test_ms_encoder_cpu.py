"""Multistream encoder, host side (no GPU needed): the argument rules of opus_multistream_encoder_get_size / _create / _init and
of the surround variants, the ctl rules that need no device, and the functions the device runs per packet
(csrc/opus_ms_encoder.h, ms_pack_packet of csrc/opus_multistream.h, through the host build tests/hostsim/ms_pack.cpp): layout
checks, rate allocation, byte budgets and the framing of each stream, against the plain-Python restatement in tests/ms_enc_framing.py."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import ms_enc_framing as E
import ms_framing as M
import oracle_lib as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OK, BAD_ARG, BUFFER_TOO_SMALL, UNIMPLEMENTED = 0, -1, -2, -5
LOWDELAY, AUDIO, VOIP = 2051, 2049, 2048
AUTO, BITRATE_MAX = -1000, -1
CELT_FB_20MS = 0xF8
CELT_FB_10MS = 0xF0
CELT_FB_2P5MS = 0xE0


def _lib():
    import concentus_b200 as cb
    return cb, cb.lib()


@pytest.fixture(scope="module")
def hs(tmp_path_factory):
    """tests/hostsim/ms_pack.cpp, compiled for the CPU into a temporary directory."""
    so = str(tmp_path_factory.mktemp("ms_pack") / "libms_pack.so")
    subprocess.run(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-Wno-unused-function", "-o", so,
                    os.path.join(ROOT, "tests", "hostsim", "ms_pack.cpp")], check=True)
    hs = C.CDLL(so)
    hs.hostsim_ms_pack.argtypes = [C.c_void_p, C.c_int32, C.c_int, C.c_int, C.c_void_p, C.c_int32]
    hs.hostsim_ms_check_layout.argtypes = [C.c_int, C.c_int, C.c_int, C.c_void_p]
    hs.hostsim_ms_surround_layout.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    hs.hostsim_ms_rate_allocation.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]
    return hs


def _u8(a):
    return np.ascontiguousarray(np.asarray(a, dtype=np.uint8))


def _create(L, Fs, channels, streams, coupled, mapping, app=LOWDELAY):
    err = C.c_int(99)
    m = _u8(mapping) if mapping is not None else None
    h = L.opus_multistream_encoder_create(Fs, channels, streams, coupled, O.ptr(m) if m is not None else None, app, C.byref(err))
    return h, err.value


# ---- argument rules ----

@pytest.mark.parametrize("channels,streams,coupled,mapping,want", [
    (6, 4, 2, [0, 4, 1, 2, 3, 5], OK),          # 5.1, explicit layout
    (2, 1, 1, [0, 1], OK),
    (1, 1, 0, [0], OK),
    (3, 2, 0, [0, 1, 255], OK),                  # an ignored input channel
    (3, 1, 1, [0, 1, 1], OK),                    # a stream channel fed twice: the first input is used
    (2, 1, 1, [0, 0], BAD_ARG),                  # stream channel 1 of the coupled stream has no input
    (2, 2, 0, [0, 0], BAD_ARG),                  # mono stream 1 has no input
    (2, 1, 0, [0, 1], BAD_ARG),                  # entry >= streams + coupled
    (0, 1, 0, [], BAD_ARG),
    (256, 1, 0, [0] * 256, BAD_ARG),
    (2, 0, 0, [0, 1], BAD_ARG),
    (2, 1, 2, [0, 1], BAD_ARG),                  # coupled > streams
    (2, 1, -1, [0, 1], BAD_ARG),
    (255, 254, 2, list(range(255)), BAD_ARG),    # streams > 255 - coupled
])
def test_create_init_layout_rules(hs, channels, streams, coupled, mapping, want):
    cb, L = _lib()
    mp = _u8(mapping + [0] * (256 - len(mapping)))
    assert hs.hostsim_ms_check_layout(channels, streams, coupled, O.ptr(mp)) == (0 if want == OK else BAD_ARG)
    h, err = _create(L, 48000, channels, streams, coupled, mp)
    assert err == want
    assert bool(h) == (want == OK)
    if h:
        L.opus_multistream_encoder_destroy(C.c_void_p(h))


def test_get_size_and_init_in_place():
    cb, L = _lib()
    one = L.opus_encoder_get_size(2)
    assert L.opus_multistream_encoder_get_size(0, 0) == 0
    assert L.opus_multistream_encoder_get_size(1, 2) == 0
    assert L.opus_multistream_encoder_get_size(2, -1) == 0
    s4 = L.opus_multistream_encoder_get_size(4, 2)
    s1 = L.opus_multistream_encoder_get_size(1, 0)
    assert s4 - s1 == 3 * one and s1 > one
    buf = (C.c_uint8 * s4)()
    mp = _u8([0, 4, 1, 2, 3, 5])
    assert L.opus_multistream_encoder_init(buf, 48000, 6, 4, 2, O.ptr(mp), LOWDELAY) == OK
    assert L.opus_multistream_encoder_init(buf, 48000, 6, 4, 2, O.ptr(mp), LOWDELAY) == OK   # a live block, again
    assert L.opus_multistream_encoder_init(buf, 44100, 6, 4, 2, O.ptr(mp), LOWDELAY) == BAD_ARG
    assert L.opus_multistream_encoder_init(buf, 48000, 6, 4, 2, O.ptr(mp), 1234) == BAD_ARG
    assert L.opus_multistream_encoder_init(buf, 48000, 6, 4, 2, None, LOWDELAY) == BAD_ARG
    for Fs in (8000, 12000, 16000, 24000, 48000):
        assert L.opus_multistream_encoder_init(buf, Fs, 6, 4, 2, O.ptr(mp), AUDIO) == OK


@pytest.mark.parametrize("channels,family,want", [
    (1, 0, (OK, 1, 0, [0])), (2, 0, (OK, 1, 1, [0, 1])), (3, 0, (UNIMPLEMENTED,)),
    (1, 1, (OK, 1, 0, [0])), (2, 1, (OK, 1, 1, [0, 1])),
    (3, 1, (UNIMPLEMENTED,)), (6, 1, (UNIMPLEMENTED,)), (8, 1, (UNIMPLEMENTED,)), (9, 1, (UNIMPLEMENTED,)),
    (5, 255, (OK, 5, 0, [0, 1, 2, 3, 4])), (1, 255, (OK, 1, 0, [0])),
    (2, 2, (UNIMPLEMENTED,)), (2, 254, (UNIMPLEMENTED,)),
    (0, 0, (BAD_ARG,)), (256, 255, (BAD_ARG,)),
])
def test_surround_families(hs, channels, family, want):
    cb, L = _lib()
    st, cp = C.c_int(-7), C.c_int(-7)
    mp = np.full(256, 77, dtype=np.uint8)
    assert hs.hostsim_ms_surround_layout(channels, family, C.byref(st), C.byref(cp), O.ptr(mp)) == want[0]
    size = L.opus_multistream_surround_encoder_get_size(channels, family)
    err = C.c_int(99)
    mp2 = np.full(256, 77, dtype=np.uint8)
    st2, cp2 = C.c_int(-7), C.c_int(-7)
    h = L.opus_multistream_surround_encoder_create(48000, channels, family, C.byref(st2), C.byref(cp2), O.ptr(mp2), LOWDELAY, C.byref(err))
    assert err.value == want[0]
    if want[0] != OK:
        assert size == 0 and not h
        return
    _, streams, coupled, mapping = want
    assert (st.value, cp.value, list(mp[:channels])) == (streams, coupled, mapping)
    assert (st2.value, cp2.value, list(mp2[:channels])) == (streams, coupled, mapping)
    assert size == L.opus_multistream_encoder_get_size(streams, coupled)
    buf = (C.c_uint8 * size)()
    st3, cp3 = C.c_int(0), C.c_int(0)
    mp3 = np.zeros(256, dtype=np.uint8)
    assert L.opus_multistream_surround_encoder_init(buf, 48000, channels, family, C.byref(st3), C.byref(cp3), O.ptr(mp3), LOWDELAY) == OK
    assert (st3.value, cp3.value) == (streams, coupled)
    L.opus_multistream_encoder_destroy(C.c_void_p(h))


# ---- ctl rules (host-current blocks: no device involved) ----

def _ctl(L, h, req, *args):
    return L.opus_multistream_encoder_ctl(C.c_void_p(h), req, *args)


def test_ctl_rules():
    cb, L = _lib()
    h, err = _create(L, 48000, 6, 4, 2, [0, 4, 1, 2, 3, 5])
    assert err == OK
    v = C.c_int32(0)
    # OPUS_SET_BITRATE: stored at the multistream level, negative values refused except OPUS_AUTO / OPUS_BITRATE_MAX
    for b, want in ((256000, OK), (0, OK), (AUTO, OK), (BITRATE_MAX, OK), (-2, BAD_ARG), (-999, BAD_ARG), (10 ** 8, OK)):
        assert _ctl(L, h, 4002, C.c_int32(b)) == want
    # OPUS_GET_BITRATE: the sum of the streams' bitrates (each stream still OPUS_AUTO: 60*Fs/(Fs/400) + Fs*channels)
    assert _ctl(L, h, 4003, C.byref(v)) == OK
    assert v.value == 2 * (24000 + 96000) + 2 * (24000 + 48000)
    assert _ctl(L, h, 4003, None) == BAD_ARG
    assert _ctl(L, h, 4031, C.byref(v)) == OK and v.value == 0
    # SETs go to every stream, GETs come from stream 0
    assert _ctl(L, h, 4010, C.c_int32(3)) == OK
    enc = C.c_void_p(0)
    for s in range(4):
        assert _ctl(L, h, 5120, C.c_int32(s), C.byref(enc)) == OK and enc.value
        assert L.opus_encoder_ctl(enc, 4011, C.byref(v)) == OK and v.value == 3
    assert _ctl(L, h, 5120, C.c_int32(4), C.byref(enc)) == BAD_ARG
    assert _ctl(L, h, 5120, C.c_int32(-1), C.byref(enc)) == BAD_ARG
    _ctl(L, h, 5120, C.c_int32(0), C.byref(enc))
    assert L.opus_encoder_ctl(enc, 4010, C.c_int32(7)) == OK
    assert _ctl(L, h, 4011, C.byref(v)) == OK and v.value == 7
    assert _ctl(L, h, 4010, C.c_int32(11)) == BAD_ARG
    assert _ctl(L, h, 4006, C.c_int32(0)) == OK and _ctl(L, h, 4007, C.byref(v)) == OK and v.value == 0
    assert _ctl(L, h, 4029, C.byref(v)) == OK and v.value == 48000
    assert _ctl(L, h, 4027, C.byref(v)) == OK and v.value == 120
    # OPUS_SET_FORCE_CHANNELS(2): the coupled streams accept it, the first mono stream refuses and the loop stops there
    assert _ctl(L, h, 4022, C.c_int32(2)) == BAD_ARG
    for s, want in ((0, 2), (1, 2), (2, -1000), (3, -1000)):
        _ctl(L, h, 5120, C.c_int32(s), C.byref(enc))
        assert L.opus_encoder_ctl(enc, 4023, C.byref(v)) == OK and v.value == want
    assert _ctl(L, h, 4028) == OK
    assert _ctl(L, h, 10024, C.c_int32(1)) == UNIMPLEMENTED   # OPUS_SET_LFE: no LFE streams
    assert _ctl(L, h, 4034, C.c_int32(0)) == UNIMPLEMENTED    # a decoder request
    assert L.opus_multistream_encoder_ctl(None, 4003, C.byref(v)) == BAD_ARG
    L.opus_multistream_encoder_destroy(C.c_void_p(h))


def test_encode_argument_errors():
    """Decided before anything is coded, so no device is involved."""
    cb, L = _lib()
    h, err = _create(L, 48000, 6, 4, 2, [0, 4, 1, 2, 3, 5])
    pcm = np.zeros(2880 * 6, dtype=np.int16)
    out = np.zeros(8000, dtype=np.uint8)
    for fs in (0, 100, 480 * 3, 959, 2880 * 2):
        assert L.opus_multistream_encode(C.c_void_p(h), O.ptr(pcm), fs, O.ptr(out), 4000) == BAD_ARG
    assert L.opus_multistream_encode(C.c_void_p(h), O.ptr(pcm), 960, O.ptr(out), 4 * 4 - 2) == BUFFER_TOO_SMALL
    assert L.opus_multistream_encode(C.c_void_p(h), O.ptr(pcm), 960, O.ptr(out), 0) == BAD_ARG
    # OPUS_SET_EXPERT_FRAME_DURATION goes to every stream: 10 ms of a 20 ms call is an argument error, as in opus_encode spans
    assert _ctl(L, h, 4040, C.c_int32(5003)) == OK
    assert L.opus_multistream_encode(C.c_void_p(h), O.ptr(pcm), 960, O.ptr(out), 4000) == BAD_ARG
    L.opus_multistream_encoder_destroy(C.c_void_p(h))


# ---- rate allocation and budgets ----

@pytest.mark.parametrize("B,channels,streams,coupled,Fs,fs", [
    (256000, 6, 4, 2, 48000, 960), (AUTO, 6, 4, 2, 48000, 960), (BITRATE_MAX, 6, 4, 2, 48000, 960), (64000, 2, 1, 1, 48000, 120),
    (32000, 1, 1, 0, 16000, 320), (500, 8, 5, 3, 48000, 2880), (0, 3, 3, 0, 24000, 480), (2000000, 2, 2, 0, 8000, 160),
    (96000, 2, 1, 1, 48000, 240), (48000, 5, 5, 0, 12000, 120), (AUTO, 1, 1, 0, 8000, 480), (10 ** 9, 6, 4, 2, 48000, 960),
])
def test_rate_allocation(hs, B, channels, streams, coupled, Fs, fs):
    got = np.zeros(streams, dtype=np.int32)
    hs.hostsim_ms_rate_allocation(B, channels, streams, coupled, Fs, fs, O.ptr(got))
    want = [max(-2 ** 31, min(2 ** 31 - 1, r)) for r in E.ms_rates(B, channels, streams, coupled, Fs, fs)]
    assert list(got) == want


def test_rate_allocation_worked_examples(hs):
    got = np.zeros(4, dtype=np.int32)
    hs.hostsim_ms_rate_allocation(256000, 6, 4, 2, 48000, 960, O.ptr(got))
    assert list(got) == [78666, 78666, 49333, 49333]
    one = np.zeros(1, dtype=np.int32)
    for B, ch, cp in ((96000, 2, 1), (64000, 2, 1), (48000, 1, 0), (256000, 2, 1), (32000, 1, 0)):
        hs.hostsim_ms_rate_allocation(B, ch, 1, cp, 48000, 960, O.ptr(one))
        assert B - 1 <= one[0] <= B    # a one-stream encoder gets the multistream bitrate (up to truncation on stereo)


@pytest.mark.parametrize("max_bytes,S", [(15, 4), (6144, 4), (5110, 4), (1276, 1), (100, 1), (20000, 8), (40, 8), (3, 1)])
def test_budgets(hs, max_bytes, S):
    assert hs.hostsim_ms_min_bytes(S) == 4 * S - 1
    for s in range(S):
        for tot in (0, 1, 7, 300, 1278 * s, max_bytes - 4 * (S - s) + 1):
            assert hs.hostsim_ms_stream_budget(max_bytes, tot, S, s) == E.ms_budget(max_bytes, tot, S, s)
    for B in (AUTO, BITRATE_MAX, 0, 6000, 256000, 10 ** 6):
        for fs in (120, 480, 960, 2880):
            assert hs.hostsim_ms_cbr_max_bytes(max_bytes, B, 48000, fs) == E.ms_cbr_max_bytes(max_bytes, B, 48000, fs)
    assert hs.hostsim_ms_cbr_last_bitrate(640, 48000, 960) == 640 * 400


def test_merged_schedule_bound():
    """At max_data_bytes = 1278*S - 2 every stream's budget is >= 1276 whatever the earlier streams took (each at most 1278 bytes
    after framing): the condition of the merged schedule."""
    for S in range(1, 9):
        mx = 1278 * S - 2
        for s in range(S):
            assert E.ms_budget(mx, 1278 * s, S, s) >= 1276
        if S > 1:
            assert E.ms_budget(mx - 1, 1278 * (S - 1), S, S - 1) < 1276


# ---- framing of one stream ----

def _pack(hs, pkt, sd, pad, maxlen):
    src = np.frombuffer(bytes(pkt), dtype=np.uint8).copy()
    out = np.full(maxlen + 64, 0xAA, dtype=np.uint8)
    r = hs.hostsim_ms_pack(O.ptr(src), len(pkt), int(sd), int(pad), O.ptr(out), maxlen)
    if r >= 0:
        assert (out[r:] == 0xAA).all(), "wrote past the packet"
    return r, bytes(out[:max(r, 0)])


def _frames(rng, count, size=None, sizes=None):
    if sizes is None:
        sizes = [size] * count
    return [bytes(rng.integers(0, 256, n, dtype=np.uint8)) for n in sizes]


def _cases():
    rng = np.random.default_rng(11)
    out = []
    out.append(M.build(CELT_FB_20MS, 0, _frames(rng, 1, 100)))
    out.append(M.build(CELT_FB_20MS, 0, _frames(rng, 1, 300)))                       # 2-byte self-delimiting length
    out.append(M.build(CELT_FB_10MS, 1, _frames(rng, 2, 80)))
    out.append(M.build(CELT_FB_10MS, 2, _frames(rng, 2, sizes=[60, 90])))
    out.append(M.build(CELT_FB_10MS, 2, _frames(rng, 2, sizes=[400, 90])))            # 2-byte code-2 length
    out.append(M.build(CELT_FB_20MS, 3, _frames(rng, 3, 50)))                         # code 3 CBR
    out.append(M.build(CELT_FB_20MS, 3, _frames(rng, 3, sizes=[50, 260, 70])))        # code 3 VBR
    out.append(M.build(CELT_FB_2P5MS, 3, _frames(rng, 4, sizes=[10, 10, 10, 12])))
    out.append(M.pad_packet(M.build(CELT_FB_20MS, 0, _frames(rng, 1, 100)), 40))      # padded: the padding is dropped
    out.append(M.pad_packet(M.build(CELT_FB_20MS, 0, _frames(rng, 1, 100)), 600))
    out.append(M.pad_packet(M.build(CELT_FB_10MS, 2, _frames(rng, 2, sizes=[30, 31])), 3))
    out.append(M.build(CELT_FB_10MS, 3, _frames(rng, 2, 80)))                         # code 3 of 2 equal frames -> code 1
    out.append(M.build(CELT_FB_20MS, 0, _frames(rng, 1, 1)))
    return out


@pytest.mark.parametrize("k", range(13))
@pytest.mark.parametrize("sd,pad", [(1, 0), (0, 0), (0, 1)])
def test_pack_matches_repacketizer(hs, k, sd, pad):
    pkt = _cases()[k]
    for maxlen in (len(pkt) + 3, len(pkt) + 300, 1278, 3000):
        want = E.ms_frame(pkt, sd, pad, maxlen)
        r, got = _pack(hs, pkt, sd, pad, maxlen)
        if isinstance(want, int):
            assert r == want
            continue
        assert r == len(want) and got == want
        if pad:
            assert r == maxlen   # CBR: the last stream fills the packet (padding of any size)
        # the result carries the same frames
        if not sd:
            assert M.parse(got)[2] == M.parse(pkt)[2]


def test_pack_buffer_too_small(hs):
    rng = np.random.default_rng(3)
    pkt = M.build(CELT_FB_20MS, 3, _frames(rng, 3, sizes=[50, 260, 70]))
    need = len(E.ms_frame(pkt, 1))
    assert _pack(hs, pkt, 1, 0, need)[0] == need
    assert _pack(hs, pkt, 1, 0, need - 1)[0] == BUFFER_TOO_SMALL
    assert _pack(hs, pkt, 0, 1, need - 3)[0] == BUFFER_TOO_SMALL
    assert _pack(hs, b"\xf8", 0, 0, 10)[0] == 1   # a bare TOC (a zero-length frame)
    assert _pack(hs, b"", 0, 0, 10)[0] < 0


def test_ms_packet_round_trip(hs):
    """Framed streams concatenate to a multistream packet the decoder's split takes apart into the original frames."""
    cases = _cases()
    subs = [cases[0], cases[3], cases[6], cases[9]]
    blob = b"".join(_pack(hs, p, i < len(subs) - 1, 0, 4000)[1] for i, p in enumerate(subs))
    assert blob == M.ms_packet([M.build(M.parse(p)[0] & 0xFC, *_canon(p)) for p in subs])


def _canon(p):
    """(code, frames) of the cheapest framing of p's frames, as the repacketizer picks it."""
    frames = M.parse(p)[2]
    lens = [len(f) for f in frames]
    code = 0 if len(frames) == 1 else (1 if len(frames) == 2 and lens[0] == lens[1] else (2 if len(frames) == 2 else 3))
    return code, frames

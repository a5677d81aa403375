"""Multistream decoder, host side (no GPU needed): the argument rules of opus_multistream_decoder_get_size / _create / _init /
_ctl (libopus opus_multistream.h), and the packet split the device runs per multistream packet (csrc/opus_multistream.h, through
the host simulation tests/hostsim): validation codes, and undelimited sub-packets that parse to the source's frames."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import ms_framing as M
import oracle_lib as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OK, BAD_ARG, BUFFER_TOO_SMALL, INVALID_PACKET, UNIMPLEMENTED = 0, -1, -2, -4, -5
CELT_FB_20MS = 0xF8     # CELT-only, fullband, 20 ms (config 31)
CELT_FB_10MS = 0xF0     # config 30
CELT_FB_2P5MS = 0xE0    # config 28
SILK_WB_20MS = 0x48     # SILK-only, wideband, 20 ms (config 9)


def _lib():
    import concentus_b200 as cb
    return cb, cb.lib()


@pytest.fixture(scope="module")
def hs(tmp_path_factory):
    """tests/hostsim/ms_split.cpp, compiled for the CPU into a temporary directory."""
    so = str(tmp_path_factory.mktemp("ms_split") / "libms_split.so")
    subprocess.run(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-Wno-unused-function", "-o", so,
                    os.path.join(ROOT, "tests", "hostsim", "ms_split.cpp")], check=True)
    hs = C.CDLL(so)
    hs.hostsim_ms_split.argtypes = [C.c_void_p, C.c_int32, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    return hs


def _split(hs, pkt, S, frame_size=5760, Fs=48000, length=None):
    src = np.frombuffer(bytes(pkt) + b"\0", dtype=np.uint8).copy()
    out = np.zeros(len(src) + 1, dtype=np.uint8)
    eo = np.zeros(S, dtype=np.int64)
    el = np.zeros(S, dtype=np.int32)
    n = len(pkt) if length is None else length
    r = hs.hostsim_ms_split(O.ptr(src), n, S, Fs, frame_size, O.ptr(out), O.ptr(eo), O.ptr(el))
    return r, out, eo, el


def _lib_parse(L, pkt):
    """The library's opus_packet_parse: (count, toc, frames)."""
    a = np.frombuffer(bytes(pkt) + b"\0", dtype=np.uint8).copy()
    toc = C.c_ubyte(0)
    sizes = (C.c_int16 * 48)()
    off = C.c_int(0)
    L.opus_packet_parse.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    n = L.opus_packet_parse(O.ptr(a), len(pkt), C.byref(toc), None, sizes, C.byref(off))
    if n < 0:
        return n, None, None
    frames, p = [], off.value
    for i in range(n):
        frames.append(bytes(a[p:p + sizes[i]]))
        p += sizes[i]
    return n, toc.value, frames


def test_multistream_argument_rules_and_ctl():
    cb, L = _lib()
    gs = L.opus_multistream_decoder_get_size
    assert gs(0, 0) == 0 and gs(1, 2) == 0 and gs(2, -1) == 0 and gs(-1, 0) == 0
    assert gs(1, 0) > 0 and gs(4, 2) >= 4 * L.opus_decoder_get_size(2) and gs(255, 0) > 0
    err = C.c_int(0)
    ident = np.arange(255, dtype=np.uint8)

    def create(Fs, ch, S, cpl, mapping):
        m = np.asarray(mapping, dtype=np.uint8)
        h = L.opus_multistream_decoder_create(Fs, ch, S, cpl, O.ptr(m), C.byref(err))
        if h:
            L.opus_multistream_decoder_destroy(C.c_void_p(h))
        return err.value, bool(h)
    # create / init: channels 1..255, 0 <= coupled <= streams, streams >= 1, streams <= 255 - coupled, mapping < streams+coupled or 255
    for args in ((48000, 0, 1, 0, [0]), (48000, 256, 1, 0, ident), (48000, 2, 1, 2, [0, 1]), (48000, 1, 0, 0, [0]),
                 (48000, 1, 1, -1, [0]), (48000, 1, 200, 56, [0]), (48000, 2, 1, 0, [0, 1]), (48000, 3, 2, 1, [0, 3, 1]),
                 (44100, 2, 1, 1, [0, 1]), (96000, 1, 1, 0, [0])):
        assert create(*args) == (BAD_ARG, False), args
    for args in ((48000, 1, 1, 0, [0]), (8000, 2, 1, 1, [1, 0]), (24000, 3, 2, 1, [0, 2, 255]), (48000, 4, 1, 0, [0, 0, 255, 0]),
                 (16000, 255, 255, 0, ident), (48000, 2, 128, 127, [0, 254]), (12000, 6, 4, 2, [0, 4, 1, 2, 3, 5])):
        assert create(*args) == (OK, True), args
    # init on caller memory, also re-initialised in place
    buf = (C.c_uint8 * gs(4, 2))()
    m51 = np.array([0, 4, 1, 2, 3, 5], dtype=np.uint8)
    assert L.opus_multistream_decoder_init(buf, 48000, 6, 4, 2, O.ptr(m51)) == OK
    assert L.opus_multistream_decoder_init(buf, 48000, 6, 4, 2, O.ptr(m51)) == OK
    assert L.opus_multistream_decoder_init(buf, 48000, 6, 4, 3, O.ptr(m51)) == OK   # 3 coupled + 1 mono, mapping still valid
    assert L.opus_multistream_decoder_init(buf, 48000, 6, 4, 2, O.ptr(np.array([0, 6, 1, 2, 3, 5], dtype=np.uint8))) == BAD_ARG
    assert L.opus_multistream_decoder_init(buf, 48000, 6, 4, 2, O.ptr(m51)) == OK
    h = C.c_void_p(C.addressof(buf))
    ctl = L.opus_multistream_decoder_ctl
    v, u = C.c_int32(0), C.c_uint32(7)
    assert ctl(h, cb.OPUS_GET_SAMPLE_RATE_REQUEST, C.byref(v)) == OK and v.value == 48000
    assert ctl(h, cb.OPUS_GET_BANDWIDTH_REQUEST, C.byref(v)) == OK and v.value == 0
    assert ctl(h, cb.OPUS_GET_LAST_PACKET_DURATION_REQUEST, C.byref(v)) == OK and v.value == 0
    assert ctl(h, cb.OPUS_GET_FINAL_RANGE_REQUEST, C.byref(u)) == OK and u.value == 0
    assert ctl(h, cb.OPUS_SET_GAIN_REQUEST, C.c_int32(40000)) == BAD_ARG
    assert ctl(h, cb.OPUS_SET_GAIN_REQUEST, C.c_int32(-1234)) == OK
    assert ctl(h, cb.OPUS_GET_GAIN_REQUEST, C.byref(v)) == OK and v.value == -1234
    assert ctl(h, cb.OPUS_GET_PITCH_REQUEST, C.byref(v)) == UNIMPLEMENTED
    assert ctl(h, 12345) == UNIMPLEMENTED
    assert ctl(h, cb.OPUS_RESET_STATE) == OK
    p = C.c_void_p(0)
    for bad in (-1, 4, 255):
        assert ctl(h, cb.OPUS_MULTISTREAM_GET_DECODER_STATE_REQUEST, C.c_int32(bad), C.byref(p)) == BAD_ARG
    dec = []
    for s in range(4):
        assert ctl(h, cb.OPUS_MULTISTREAM_GET_DECODER_STATE_REQUEST, C.c_int32(s), C.byref(p)) == OK and p.value
        dec.append(p.value)
        # the embedded block is an ordinary decoder: coupled streams are stereo, the others mono; SET_GAIN reached every stream
        assert L.opus_decoder_ctl(C.c_void_p(p.value), cb.OPUS_GET_GAIN_REQUEST, C.byref(v)) == OK and v.value == -1234
        assert L.opus_decoder_ctl(C.c_void_p(p.value), cb.OPUS_GET_SAMPLE_RATE_REQUEST, C.byref(v)) == OK and v.value == 48000
    assert dec[0] > C.addressof(buf) and len(set(np.diff(dec))) == 1 and dec[-1] < C.addressof(buf) + len(buf)
    # arguments decided before any device work
    pcm = np.zeros(960 * 6, dtype=np.int16)
    pkt = np.zeros(8, dtype=np.uint8)
    assert L.opus_multistream_decode(h, O.ptr(pkt), 8, O.ptr(pcm), 0, 0) == BAD_ARG
    assert L.opus_multistream_decode(h, O.ptr(pkt), 8, O.ptr(pcm), -960, 0) == BAD_ARG
    assert L.opus_multistream_decode(h, O.ptr(pkt), -1, O.ptr(pcm), 960, 0) == BAD_ARG
    assert L.opus_multistream_decode(h, O.ptr(pkt), 8, O.ptr(pcm), 960, 2) == BAD_ARG
    assert L.opus_multistream_decode(h, O.ptr(pkt), 8, None, 960, 0) == BAD_ARG


def _frames(rs, n, lo, hi):
    return [bytes(rs.randint(0, 256, size=rs.randint(lo, hi + 1)).astype(np.uint8)) for _ in range(n)]


def _subpackets(rs, toc_cfg):
    """Ordinary packets of every frame-count code, one- and two-byte lengths, CBR / VBR code 3, padding."""
    out = []
    out.append(M.build(toc_cfg, 0, _frames(rs, 1, 2, 200)))
    out.append(M.build(toc_cfg, 0, _frames(rs, 1, 252, 1275)))
    f = _frames(rs, 1, 2, 400)[0]
    out.append(M.build(toc_cfg, 1, [f, bytes(reversed(f))]))
    out.append(M.build(toc_cfg, 2, _frames(rs, 1, 252, 700) + _frames(rs, 1, 2, 100)))
    out.append(M.build(toc_cfg, 2, _frames(rs, 1, 0, 10) + _frames(rs, 1, 300, 900)))
    f = _frames(rs, 1, 2, 300)[0]
    out.append(M.build(toc_cfg, 3, [f] * 2))                                  # CBR
    out.append(M.build(toc_cfg, 3, [f] * 2, pad=1))                           # CBR, one padding-length byte and no padding
    out.append(M.build(toc_cfg, 3, _frames(rs, 2, 1, 400)))                   # VBR
    out.append(M.build(toc_cfg, 3, _frames(rs, 2, 250, 600), pad=300))        # VBR, two-byte lengths, 255-continued padding
    out.append(M.build(toc_cfg, 3, [bytes(40)] * 2, pad=17))
    return out


@pytest.mark.parametrize("toc_cfg,per_frame", [(CELT_FB_20MS, 960), (CELT_FB_10MS, 480), (CELT_FB_2P5MS, 120)])
def test_multistream_split_undelimits_every_framing(hs, toc_cfg, per_frame):
    cb, L = _lib()
    rs = np.random.RandomState(7 + per_frame)
    subs = _subpackets(rs, toc_cfg)
    # group sub-packets of equal duration into multistream packets of 1..5 streams, in rotating orders
    by_n = {}
    for p in subs:
        by_n.setdefault(len(M.parse(p)[2]), []).append(p)
    cases = 0
    for group in by_n.values():
        for S in range(1, 6):
            for rot in range(len(group)):
                streams = [group[(rot + k) % len(group)] for k in range(S)]
                ms = M.ms_packet(streams)
                assert len(ms) >= 2 * S - 1
                r, out, eo, el = _split(hs, ms, S)
                nfr = len(M.parse(streams[0])[2])
                assert r == nfr * per_frame, (S, rot, r)
                for s in range(S):
                    e = bytes(out[eo[s]:eo[s] + el[s]])
                    assert el[s] <= (len(ms) if s == S - 1 else len(M.self_delimit(streams[s])))
                    n, toc, frames = _lib_parse(L, e)
                    src = M.parse(streams[s])
                    assert n == len(src[2]) and toc == src[0] and frames == [bytes(x) for x in src[2]], (S, s)
                    if s < S - 1:
                        assert e[0] & 3 == streams[s][0] & 3   # same frame-count code, no padding
                        assert not (e[0] & 3 == 3 and e[1] & 0x40)
                    else:
                        assert e == bytes(streams[s])          # the last stream is used as it is
                # the undelimited packets lie inside their sources, with the frames where they were: only headers were rewritten
                src = np.frombuffer(ms, dtype=np.uint8)
                pos = 0
                for s in range(S):
                    n_sd = len(M.self_delimit(streams[s])) if s < S - 1 else len(streams[s])
                    assert pos <= eo[s] and eo[s] + el[s] <= pos + n_sd
                    hdr = el[s] - sum(len(f) for f in M.parse(streams[s])[2])
                    assert np.array_equal(out[eo[s] + hdr:eo[s] + el[s]], src[eo[s] + hdr:eo[s] + el[s]])
                    pos += n_sd
                cases += 1
    assert cases > 20


def test_multistream_split_rejections(hs):
    _, L = _lib()
    rs = np.random.RandomState(3)
    a = M.build(CELT_FB_20MS, 0, _frames(rs, 1, 300, 400))        # 20 ms, two-byte self-delimited length
    b = M.build(CELT_FB_20MS, 3, _frames(rs, 2, 10, 60))          # 40 ms
    c = M.build(CELT_FB_10MS, 1, [bytes(30)] * 2)                  # 20 ms as two 10 ms frames
    d = M.build(CELT_FB_20MS, 0, _frames(rs, 1, 5, 50))

    def check(pkt, S, want, frame_size=5760, length=None):
        r, out, eo, el = _split(hs, pkt, S, frame_size, length=length)
        assert r == want, (want, r)
        if want < 0:
            # every stream gets the reject marker: a packet that the decoder stages refuse to parse, so no state is touched
            for s in range(S):
                assert el[s] > 0 and _lib_parse(L, bytes(out[eo[s]:eo[s] + el[s]]))[0] == INVALID_PACKET
        elif want == 0:
            assert (el == 0).all()
        return el
    check(M.ms_packet([a, c, d]), 3, 960)
    check(M.ms_packet([a, c, d]), 3, 960, frame_size=960)
    check(b"", 3, 0)                                               # lost: every stream conceals
    check(M.ms_packet([a, d]), 2, BAD_ARG, length=-1)
    check(M.ms_packet([a, c, d]), 3, INVALID_PACKET, length=4)     # len < 2S-1
    check(bytes([CELT_FB_20MS, 1, 0x55]), 2, INVALID_PACKET)       # nothing left for the last stream
    check(M.ms_packet([a, b]), 2, INVALID_PACKET)                  # 20 ms and 40 ms
    check(M.ms_packet([d, a, b]), 3, INVALID_PACKET)
    check(M.ms_packet([a, d]), 2, BUFFER_TOO_SMALL, frame_size=959)
    check(M.ms_packet([b, b]), 2, BUFFER_TOO_SMALL, frame_size=1919)
    check(M.ms_packet([b, b]), 2, 1920, frame_size=1920)
    # truncated / garbled self-delimited length: it claims more bytes than the packet has
    ms = bytearray(M.ms_packet([a, d]))
    check(bytes(ms[:200]), 2, INVALID_PACKET)
    ms[1] = 255; ms[2] = 255
    check(bytes(ms), 2, INVALID_PACKET)
    bad_cbr = bytearray(M.ms_packet([c, d]))   # code 1: both frames take the self-delimited length
    bad_cbr[1] = 250
    check(bytes(bad_cbr), 2, INVALID_PACKET)
    # a parse error comes before a duration mismatch or a size check of a later stream
    check(bytes(ms) + M.ms_packet([b]), 2, INVALID_PACKET, frame_size=100)
    # SILK with a frame in stream 1: outside this decoder's scope, decided before anything is decoded ...
    silk = M.build(SILK_WB_20MS, 0, _frames(rs, 1, 20, 40))
    check(M.ms_packet([a, silk, d]), 3, UNIMPLEMENTED)
    # ... but only after the validation, whose codes come first
    check(M.ms_packet([a, silk, d]), 3, BUFFER_TOO_SMALL, frame_size=480)
    # a SILK TOC whose frames are empty is concealment in CELT and accepted
    check(M.ms_packet([a, M.build(SILK_WB_20MS, 0, [b"\x00"]), d]), 3, 960)
    # trailing bytes belong to the last stream
    ms = M.ms_packet([a, d]) + bytes(7)
    r, out, eo, el = _split(hs, ms, 2)
    assert r == 960 and el[1] == len(d) + 7
    n, _, frames = _lib_parse(L, bytes(out[eo[1]:eo[1] + el[1]]))
    assert n == 1 and len(frames[0]) == len(d) - 1 + 7

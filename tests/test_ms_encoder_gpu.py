"""Multistream encoder on the GPU (opus_multistream_encode, _span, _span_device).  The reference multistream encoder is per-stream
opus_encode_native with a rate allocation, byte budgets and repacketizer framing around it, so it is pinned two ways: one-stream
layouts against the reference's packets and final ranges of the golden fixtures (tests/golden/enc_*.npz), and any layout against
fresh single-stream encoders of this library — which the rest of the suite pins to the reference — driven frame by frame and stream
by stream with the bitrates and budgets of libopus's encode loop (restated in tests/ms_enc_framing.py) and framed in plain Python."""
import ctypes as C
import glob
import os

import numpy as np
import pytest

import ms_enc_framing as E
import ms_framing as M
import oracle_lib as O

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
OK, BAD_ARG, BUFFER_TOO_SMALL, UNIMPLEMENTED = 0, -1, -2, -5
LOWDELAY, AUDIO = 2051, 2049
AUTO = -1000
SET_BITRATE, GET_BITRATE, SET_VBR, GET_VBR, SET_CVBR, SET_COMPLEXITY = 4002, 4003, 4006, 4007, 4020, 4010
GET_APPLICATION, SET_APPLICATION, GET_FINAL_RANGE, RESET = 4001, 4000, 4031, 4028
MAP_51 = [0, 4, 1, 2, 3, 5]


def _cb():
    import concentus_b200 as cb
    assert cb.lib().opus_b200_init(0) == 0, "CUDA device required: no CPU fallback exists"
    return cb


def _get(L, h, req, ms=True):
    v = C.c_int32(0)
    f = L.opus_multistream_encoder_ctl if ms else L.opus_encoder_ctl
    assert f(C.c_void_p(h), req, C.byref(v)) == OK
    return v.value & 0xFFFFFFFF if req == GET_FINAL_RANGE else v.value


def _stream(L, h, s):
    p = C.c_void_p(0)
    assert L.opus_multistream_encoder_ctl(C.c_void_p(h), 5120, C.c_int32(s), C.byref(p)) == OK
    return p.value


def _signal(T, channels, seed):
    kinds = ("music", "tone", "clicks", "noise")
    cols = [O.test_signal(T, 1, seed * 31 + c, kinds[(seed + c) % 4]).reshape(T) for c in range(channels)]
    x = np.stack(cols, axis=1).astype(np.int16)
    if channels > 1:
        x[:, -1] //= 4   # channels of different loudness
    return np.ascontiguousarray(x)


class Layout:
    def __init__(self, Fs, channels, S, coupled, mapping, app=LOWDELAY, bitrate=AUTO, vbr=1, cvbr=1, complexity=9, stream_app=None):
        self.Fs, self.channels, self.S, self.coupled, self.mapping = Fs, channels, S, coupled, list(mapping)
        self.app, self.bitrate, self.vbr, self.cvbr, self.complexity = app, bitrate, vbr, cvbr, complexity
        self.stream_app = stream_app or {}   # stream -> application set through OPUS_MULTISTREAM_GET_ENCODER_STATE

    def create(self, L):
        m = np.array(self.mapping, dtype=np.uint8)
        err = C.c_int(0)
        h = L.opus_multistream_encoder_create(self.Fs, self.channels, self.S, self.coupled, O.ptr(m), self.app, C.byref(err))
        assert h and err.value == OK, err.value
        for req, v in ((SET_BITRATE, self.bitrate), (SET_VBR, self.vbr), (SET_CVBR, self.cvbr), (SET_COMPLEXITY, self.complexity)):
            assert L.opus_multistream_encoder_ctl(C.c_void_p(h), req, C.c_int32(v)) == OK
        for s, a in self.stream_app.items():
            assert L.opus_encoder_ctl(C.c_void_p(_stream(L, h, s)), SET_APPLICATION, C.c_int32(a)) == OK
        return h

    def sources(self):
        ks = [(2 * s, 2 * s + 1) if s < self.coupled else (self.coupled + s,) for s in range(self.S)]
        return [[self.mapping.index(k) for k in kk] for kk in ks]


class Model:
    """libopus's multistream encode loop over fresh single-stream encoders of this library."""

    def __init__(self, L, lay):
        self.L, self.lay = L, lay
        self.enc = []
        for s in range(lay.S):
            err = C.c_int(0)
            app = lay.stream_app.get(s, lay.app)
            h = L.opus_encoder_create(lay.Fs, 2 if s < lay.coupled else 1, app, C.byref(err))
            assert h
            for req, v in ((SET_VBR, lay.vbr), (SET_CVBR, lay.cvbr), (SET_COMPLEXITY, lay.complexity)):
                assert L.opus_encoder_ctl(C.c_void_p(h), req, C.c_int32(v)) == OK
            self.enc.append(h)

    def encode(self, pcm, fs, max_data_bytes):
        L, lay = self.L, self.lay
        S = lay.S
        if max_data_bytes < 4 * S - 1:
            return BUFFER_TOO_SMALL, b""
        rates = E.ms_rates(lay.bitrate, lay.channels, S, lay.coupled, lay.Fs, fs)
        for s in range(S):
            L.opus_encoder_ctl(C.c_void_p(self.enc[s]), SET_BITRATE, C.c_int32(rates[s]))
        cbr = not lay.vbr
        mx = E.ms_cbr_max_bytes(max_data_bytes, lay.bitrate, lay.Fs, fs) if cbr else max_data_bytes
        out, tot = b"", 0
        buf = np.zeros(1276, dtype=np.uint8)
        for s, src in enumerate(lay.sources()):
            x = np.ascontiguousarray(pcm[:, src])
            curr = E.ms_budget(mx, tot, S, s)
            if cbr and s == S - 1:
                L.opus_encoder_ctl(C.c_void_p(self.enc[s]), SET_BITRATE, C.c_int32(curr * (8 * lay.Fs // fs)))
            r = L.opus_encode(C.c_void_p(self.enc[s]), O.ptr(x), fs, O.ptr(buf), min(curr, 1276))
            if r < 0:
                return r, b""
            p = E.ms_frame(bytes(buf[:r]), s < S - 1, cbr and s == S - 1, mx - tot)
            assert not isinstance(p, int)
            out += p
            tot += len(p)
        return tot, out

    def final_range(self):
        r = 0
        for h in self.enc:
            r ^= _get(self.L, h, GET_FINAL_RANGE, ms=False)
        return r

    def bitrate(self):
        return sum(_get(self.L, h, GET_BITRATE, ms=False) for h in self.enc)

    def close(self):
        for h in self.enc:
            self.L.opus_encoder_destroy(C.c_void_p(h))


def _span(L, hs, pcm, F, fs, mx, device=False):
    """pcm [n, F*fs, channels] -> (packets [n, F] bytes, rets [n, F])."""
    n = len(hs)
    arr = (C.c_void_p * n)(*hs)
    x = np.ascontiguousarray(pcm, dtype=np.int16)
    if device:
        import torch
        dx = torch.from_numpy(x.reshape(-1)).cuda()
        dd = torch.zeros(n * F * mx, dtype=torch.uint8, device="cuda")
        dr = torch.zeros(n * F, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()   # the library's stream does not wait for torch's
        assert L.opus_multistream_encode_span_device(arr, n, F, C.c_void_p(dx.data_ptr()), fs, C.c_void_p(dd.data_ptr()), mx,
                                                     C.c_void_p(dr.data_ptr())) == OK
        assert L.opus_b200_enc_synchronize() == OK
        data, rets = dd.cpu().numpy().reshape(n * F, mx), dr.cpu().numpy()
    else:
        data = np.zeros((n * F, mx), dtype=np.uint8)
        rets = np.zeros(n * F, dtype=np.int32)
        assert L.opus_multistream_encode_span(arr, n, F, O.ptr(x), fs, O.ptr(data), mx, O.ptr(rets)) == OK
    pk = [[bytes(data[m * F + f, :max(rets[m * F + f], 0)]) for f in range(F)] for m in range(n)]
    return pk, rets.reshape(n, F)


def _scalar(L, h, pcm, fs, mx):
    out = np.zeros(mx, dtype=np.uint8)
    x = np.ascontiguousarray(pcm, dtype=np.int16)
    r = L.opus_multistream_encode(C.c_void_p(h), O.ptr(x), fs, O.ptr(out), mx)
    return r, bytes(out[:max(r, 0)])


# ---- 1. reference pin: one-stream layouts on the golden fixtures ----

GOLDEN_ENC = sorted(glob.glob(os.path.join(GOLDEN, "enc_*.npz")))


@pytest.mark.parametrize("path", GOLDEN_ENC, ids=[os.path.basename(p)[4:-4] for p in GOLDEN_ENC])
@pytest.mark.parametrize("how", ["family0", "explicit"])
@pytest.mark.parametrize("call", ["scalar", "span", "device"])
def test_golden_one_stream(path, how, call):
    cb = _cb()
    L = cb.lib()
    z = np.load(path)
    ch, fs = int(z["channels"]), int(z["frame_size"])
    pcm, F = z["pcm"], len(z["lens"])
    if how == "family0":
        st, cp = C.c_int(0), C.c_int(0)
        mp = np.zeros(255, dtype=np.uint8)
        err = C.c_int(0)
        h = L.opus_multistream_surround_encoder_create(48000, ch, 0, C.byref(st), C.byref(cp), O.ptr(mp), LOWDELAY, C.byref(err))
        assert h and (st.value, cp.value) == (1, ch - 1)
    else:
        h = Layout(48000, ch, 1, ch - 1, list(range(ch))).create(L)
    for req, v in ((SET_BITRATE, int(z["bitrate"])), (SET_VBR, int(z["vbr"])), (SET_CVBR, int(z["cvbr"])), (SET_COMPLEXITY, int(z["complexity"]))):
        assert L.opus_multistream_encoder_ctl(C.c_void_p(h), req, C.c_int32(v)) == OK
    want = [bytes(z["data"][z["offs"][f]:z["offs"][f] + z["lens"][f]]) for f in range(F)]
    if call == "scalar":
        for f in range(F):
            r, p = _scalar(L, h, pcm[f * fs:(f + 1) * fs], fs, 1275)
            assert r == z["lens"][f] and p == want[f], f
            assert _get(L, h, GET_FINAL_RANGE) == z["enc_ranges"][f], f
    else:
        pk, rets = _span(L, [h], pcm[None, :F * fs], F, fs, 1275, device=call == "device")
        assert list(rets[0]) == list(z["lens"])
        assert pk[0] == want
        assert _get(L, h, GET_FINAL_RANGE) == z["enc_ranges"][F - 1]
    L.opus_multistream_encoder_destroy(C.c_void_p(h))


# ---- 2. composition: random layouts against single-stream encoders ----

def _random_layout(rng, Fs, app=LOWDELAY, vbr=1, cvbr=1):
    S = int(rng.integers(1, 9))
    cp = int(rng.integers(0, S + 1))
    need = list(range(S + cp))
    extra = [int(rng.integers(0, S + cp)) for _ in range(int(rng.integers(0, 3)))] + [255] * int(rng.integers(0, 2))
    mapping = need + extra
    rng.shuffle(mapping)
    mapping = [int(v) for v in mapping]
    C_ = len(mapping)
    return Layout(Fs, C_, S, cp, mapping, app=app, vbr=vbr, cvbr=cvbr, complexity=int(rng.integers(0, 11)),
                  bitrate=int(rng.choice([AUTO, 24000 * S, 48000 * S + 64000 * cp, 32000 * (S + cp)])))


CASES = [
    # (seed, Fs, frame_size, F, n, app, vbr, cvbr, max_data_bytes or None for 1278*S-2)
    (1, 48000, 960, 6, 4, LOWDELAY, 1, 0, None),      # merged
    (2, 48000, 960, 6, 4, LOWDELAY, 1, 1, 6144),
    (3, 48000, 480, 6, 3, LOWDELAY, 0, 0, 6144),      # CBR: ordered, last stream padded
    (4, 48000, 120, 8, 3, LOWDELAY, 0, 0, 2000),
    (5, 16000, 320, 5, 3, LOWDELAY, 1, 0, None),
    (6, 8000, 80, 5, 2, LOWDELAY, 0, 1, 600),
    (7, 24000, 1440, 3, 2, LOWDELAY, 1, 0, None),     # 60 ms
    (8, 12000, 480, 3, 2, LOWDELAY, 0, 0, 3000),      # 40 ms CBR
    (9, 48000, 960, 5, 3, AUDIO, 1, 1, 6144),         # AUDIO: CELT at these rates
    (10, 48000, 240, 6, 3, LOWDELAY, 1, 0, 60),       # tight: later streams shrink, some fail
    (11, 48000, 960, 4, 3, LOWDELAY, 0, 0, 40),
]


@pytest.mark.parametrize("case", CASES, ids=[str(c[0]) for c in CASES])
@pytest.mark.parametrize("device", [False, True], ids=["span", "device"])
def test_composition(case, device):
    seed, Fs, fs, F, n, app, vbr, cvbr, mx = case
    cb = _cb()
    L = cb.lib()
    rng = np.random.default_rng(seed)
    base = _random_layout(rng, Fs, app, vbr, cvbr)
    lays = []
    for m in range(n):   # one geometry, different mappings and settings per encoder
        mp = list(base.mapping)
        if m % 2:
            mp = mp[::-1]
        br = base.bitrate if m == 0 else int(rng.choice([AUTO, 20000 * base.S, 300000 * base.S, 64000 + 16000 * m]))
        if app == AUDIO:
            br = 96000 * base.S
        lays.append(Layout(Fs, base.channels, base.S, base.coupled, mp, app=app, vbr=vbr, cvbr=cvbr,
                           complexity=int(rng.integers(0, 11)), bitrate=br))
    if mx is None:
        mx = 1278 * base.S - 2
    pcm = np.stack([_signal(F * fs, base.channels, seed * 100 + m) for m in range(n)])
    hs = [l.create(L) for l in lays]
    pk, rets = _span(L, hs, pcm, F, fs, mx, device=device)
    for m, lay in enumerate(lays):
        mod = Model(L, lay)
        for f in range(F):
            r, p = mod.encode(pcm[m, f * fs:(f + 1) * fs], fs, mx)
            assert rets[m, f] == r, (m, f)
            assert pk[m][f] == p, (m, f)
        assert _get(L, hs[m], GET_FINAL_RANGE) == mod.final_range()
        assert _get(L, hs[m], GET_BITRATE) == mod.bitrate()
        mod.close()
        L.opus_multistream_encoder_destroy(C.c_void_p(hs[m]))


# ---- 3. the two schedules agree ----

def test_schedules_agree():
    cb = _cb()
    L = cb.lib()
    S, F, fs, n = 4, 8, 960, 6
    pcm = np.stack([_signal(F * fs, 6, 500 + m) for m in range(n)])
    out = []
    for mx in (1278 * S - 2, 1278 * S - 3):
        lays = [Layout(48000, 6, S, 2, MAP_51, bitrate=128000 + 32000 * m, vbr=1, cvbr=m % 2, complexity=m + 4) for m in range(n)]
        hs = [l.create(L) for l in lays]
        pipe0, leg0 = C.c_longlong(0), C.c_longlong(0)
        L.opus_b200_enc_path_counts(C.byref(pipe0), C.byref(leg0))
        out.append(_span(L, hs, pcm, F, fs, mx))
        pipe1, leg1 = C.c_longlong(0), C.c_longlong(0)
        L.opus_b200_enc_path_counts(C.byref(pipe1), C.byref(leg1))
        if mx == 1278 * S - 2:
            assert pipe1.value - pipe0.value == n * S   # merged: every stream through the pipeline
        else:
            assert leg1.value - leg0.value == n * S     # ordered: every pass on the one-kernel path
        for h in hs:
            L.opus_multistream_encoder_destroy(C.c_void_p(h))
    assert out[0][0] == out[1][0]
    assert (out[0][1] == out[1][1]).all() and (out[0][1] > 0).all()


# ---- 4. round trip through the multistream decoder ----

def test_round_trip_final_ranges():
    cb = _cb()
    L = cb.lib()
    lay = Layout(48000, 6, 4, 2, MAP_51, bitrate=256000, complexity=10)
    h = lay.create(L)
    err = C.c_int(0)
    d = L.opus_multistream_decoder_create(48000, 6, 4, 2, O.ptr(np.array(MAP_51, dtype=np.uint8)), C.byref(err))
    assert d
    fs, F = 960, 12
    x = _signal(F * fs, 6, 77)
    out = np.zeros((fs, 6), dtype=np.int16)
    rd = C.c_uint32(0)
    for f in range(F):
        r, p = _scalar(L, h, x[f * fs:(f + 1) * fs], fs, 6144)
        assert r > 0
        a = np.frombuffer(p, dtype=np.uint8).copy()
        assert L.opus_multistream_decode(C.c_void_p(d), O.ptr(a), r, O.ptr(out), fs, 0) == fs
        assert L.opus_multistream_decoder_ctl(C.c_void_p(d), GET_FINAL_RANGE, C.byref(rd)) == OK
        assert rd.value == _get(L, h, GET_FINAL_RANGE), f
    # the span's packets decode through the multistream decode span
    lays = [Layout(48000, 6, 4, 2, MAP_51, bitrate=192000 + 64000 * m) for m in range(3)]
    hs = [l.create(L) for l in lays]
    pcm = np.stack([_signal(F * fs, 6, 90 + m) for m in range(3)])
    pk, rets = _span(L, hs, pcm, F, fs, 6144)
    dec = cb.MSDecoderBatch(3, 48000, 6, 4, 2, MAP_51)
    blob, offs, lens = M.ms_blob([p for row in pk for p in row])
    _, drets = dec.decode_span(blob, offs, lens, F, fs)
    assert (drets == fs).all()
    assert (dec.final_ranges() == np.array([_get(L, hh, GET_FINAL_RANGE) for hh in hs], dtype=np.uint32)).all()
    dec.close()
    for hh in hs + [h]:
        L.opus_multistream_encoder_destroy(C.c_void_p(hh))
    L.opus_multistream_decoder_destroy(C.c_void_p(d))


# ---- 5. errors and state ----

def test_argument_errors_span():
    cb = _cb()
    L = cb.lib()
    lay = Layout(48000, 6, 4, 2, MAP_51)
    hs = [lay.create(L) for _ in range(2)]
    arr = (C.c_void_p * 2)(*hs)
    x = np.zeros(2 * 3 * 2880 * 6, dtype=np.int16)
    d = np.zeros(2 * 3 * 6144, dtype=np.uint8)
    r = np.zeros(6, dtype=np.int32)
    for fs in (100, 959, 2880 * 2):
        assert L.opus_multistream_encode_span(arr, 2, 3, O.ptr(x), fs, O.ptr(d), 6144, O.ptr(r)) == BAD_ARG
    assert L.opus_multistream_encode_span(arr, 2, 3, O.ptr(x), 960, O.ptr(d), 14, O.ptr(r)) == BUFFER_TOO_SMALL
    other = Layout(48000, 6, 5, 1, [0, 1, 2, 3, 4, 5]).create(L)
    mixed = (C.c_void_p * 2)(hs[0], other)
    assert L.opus_multistream_encode_span(mixed, 2, 3, O.ptr(x), 960, O.ptr(d), 6144, O.ptr(r)) == BAD_ARG
    dup = (C.c_void_p * 2)(hs[0], hs[0])
    assert L.opus_multistream_encode_span(dup, 2, 3, O.ptr(x), 960, O.ptr(d), 6144, O.ptr(r)) == BAD_ARG
    for h in hs + [other]:
        L.opus_multistream_encoder_destroy(C.c_void_p(h))


def test_stream_failure_mid_span():
    """Stream 1 is OPUS_APPLICATION_AUDIO at a rate where libopus picks SILK: it returns OPUS_UNIMPLEMENTED every frame; stream 0
    advances, stream 2 stays untouched, and the neighbouring encoders of the span are exact."""
    cb = _cb()
    L = cb.lib()
    fs, F = 960, 5
    lays = [Layout(48000, 3, 3, 0, [0, 1, 2], bitrate=24000, stream_app={1: AUDIO} if m == 1 else None, complexity=5) for m in range(3)]
    hs = [l.create(L) for l in lays]
    pcm = np.stack([_signal(F * fs, 3, 300 + m) for m in range(3)])
    pk, rets = _span(L, hs, pcm, F, fs, 1500)
    assert (rets[1] == UNIMPLEMENTED).all() and (rets[0] > 0).all() and (rets[2] > 0).all()
    for m, lay in enumerate(lays):
        mod = Model(L, lay)
        for f in range(F):
            r, p = mod.encode(pcm[m, f * fs:(f + 1) * fs], fs, 1500)
            assert (rets[m, f], pk[m][f]) == (r, p)
        for s in range(3):
            assert _get(L, _stream(L, hs[m], s), GET_FINAL_RANGE, ms=False) == _get(L, mod.enc[s], GET_FINAL_RANGE, ms=False)
        mod.close()
    # stream 2 of the failing encoder never coded a frame
    assert _get(L, _stream(L, hs[1], 2), GET_FINAL_RANGE, ms=False) == 0
    for h in hs:
        L.opus_multistream_encoder_destroy(C.c_void_p(h))


def test_state_memcpy_reset_sync_and_mixing():
    cb = _cb()
    L = cb.lib()
    fs, F, mx = 960, 4, 6144
    lay = Layout(48000, 6, 4, 2, MAP_51, bitrate=256000, vbr=0)   # CBR: the ordered schedule and the last stream's bitrate
    x = _signal(4 * F * fs, 6, 999)
    chunks = [x[i * F * fs:(i + 1) * F * fs] for i in range(4)]
    # all-scalar reference
    ref = lay.create(L)
    want = [_scalar(L, ref, chunks[i][f * fs:(f + 1) * fs], fs, mx) for i in range(4) for f in range(F)]
    want_range, want_rate = _get(L, ref, GET_FINAL_RANGE), _get(L, ref, GET_BITRATE)
    # span -> scalar -> span -> (sync, memcpy) -> span on the copy
    h = lay.create(L)
    got = []
    pk, rets = _span(L, [h], chunks[0][None], F, fs, mx)
    got += list(zip(rets[0], pk[0]))
    got += [_scalar(L, h, chunks[1][f * fs:(f + 1) * fs], fs, mx) for f in range(F)]
    pk, rets = _span(L, [h], chunks[2][None], F, fs, mx, device=True)
    got += list(zip(rets[0], pk[0]))
    assert L.opus_multistream_encoder_sync((C.c_void_p * 1)(h), 1) == OK
    size = L.opus_multistream_encoder_get_size(4, 2)
    copy = (C.c_uint8 * size)()
    C.memmove(copy, h, size)
    hc = C.addressof(copy)
    pk, rets = _span(L, [hc], chunks[3][None], F, fs, mx)
    got += list(zip(rets[0], pk[0]))
    assert [(int(r), p) for r, p in got] == [(int(r), p) for r, p in want]
    assert _get(L, hc, GET_FINAL_RANGE) == want_range
    assert _get(L, hc, GET_BITRATE) == want_rate
    # the embedded block of stream 3 answers opus_encoder_ctl: CBR left it at the bitrate of its last budget
    e3 = _stream(L, hc, 3)
    assert _get(L, e3, GET_BITRATE, ms=False) == _get(L, _stream(L, ref, 3), GET_BITRATE, ms=False)
    assert _get(L, e3, GET_VBR, ms=False) == 0
    # reset: the encoder codes like a fresh one
    assert L.opus_multistream_encoder_ctl(C.c_void_p(hc), RESET) == OK
    fresh = lay.create(L)
    pk1, r1 = _span(L, [hc], chunks[0][None], F, fs, mx)
    pk2, r2 = _span(L, [fresh], chunks[0][None], F, fs, mx)
    assert pk1 == pk2 and (r1 == r2).all()
    L.opus_multistream_encoder_sync((C.c_void_p * 1)(hc), 1)
    for hh in (ref, h, fresh):
        L.opus_multistream_encoder_destroy(C.c_void_p(hh))


def test_stage_times_and_batch_class():
    cb = _cb()
    L = cb.lib()
    ms = (C.c_double * 3)()
    ln = (C.c_longlong * 3)()
    L.opus_b200_ms_enc_stage_times(ms, ln, 1)
    b = cb.MSEncoderBatch(3, 48000, 6, 4, 2, MAP_51, bitrate=256000, complexity=10)
    pcm = np.concatenate([_signal(5 * 960, 6, 40 + m) for m in range(3)])
    data, rets = b.encode_span(pcm, 5, 960, 6144)
    assert (rets > 0).all()
    assert (b.bitrates() > 0).all()
    b.close()
    L.opus_b200_ms_enc_stage_times(ms, ln, 0)
    assert ln[0] == 1 and ln[2] == 1 and ln[1] == 0   # merged: one route, one pack, no budget pass
    assert ms[0] > 0 and ms[2] > 0

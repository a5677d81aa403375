"""The tests' oracle: what the reference (opus-fix FIXED_POINT libopus 1.1.2, restricted to its CELT paths) produces for an input.

TEST INFRASTRUCTURE ONLY.  Imported by tests/, __graft_entry__.smoke(), bench.py and tools/; nothing under concentus_b200/
imports this module.

The reference's sources are not part of this repository, so the results are computed by the host simulation of the codec headers
(tests/hostsim: the headers of concentus_b200/csrc compiled for the CPU with 1-lane teams).  That is a host build of the very
code the tests check, so it is not trusted on its own: every result it hands out is checked against a digest of the reference's
result for the same call, stored in tests/golden/oracle_digests.npy, and a call without a stored digest fails.  A change to the
shared headers therefore cannot move the oracle along with the code it checks.  The stored digests are those of calls the suite
had compared with the reference build (oracle/Makefile + oracle/ref_harness.c) before the oracle moved to the host simulation,
with the host and CUDA builds unchanged since.  A caller that wants a result with no reference behind it (a benchmark's input, a
randomised sweep) says so with pin=False.

New digests come from the reference build itself: with ORACLE_DIGEST_RECORD=<file> set the oracle runs on oracle/_ref/libopus_ref.so
(make -C oracle REF=<opus-fix source tree>) and appends a digest line per call; `python tests/oracle_lib.py record <file>` merges
them into the table.
"""
import ctypes as C
import hashlib
import os
import subprocess
import sys
import threading

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOSTSIM_SRC = os.path.join(ROOT, "tests", "hostsim", "hostsim.cpp")
HOSTSIM_SO = os.path.join(ROOT, "tests", "hostsim", "libhostsim.so")
REF_SO = os.path.join(ROOT, "oracle", "_ref", "libopus_ref.so")
DIGESTS = os.path.join(ROOT, "tests", "golden", "oracle_digests.npy")
# Set to a file path to run the oracle on the reference build and append the digest of every call there (see record() below).
RECORD = os.environ.get("ORACLE_DIGEST_RECORD")

OPUS_APPLICATION_VOIP = 2048
OPUS_APPLICATION_AUDIO = 2049
OPUS_APPLICATION_RESTRICTED_LOWDELAY = 2051
OPUS_UNIMPLEMENTED = -5


class RefEncCfg(C.Structure):
    _fields_ = [(n, C.c_int) for n in
                ("application", "bitrate", "vbr", "cvbr", "complexity", "max_bytes", "force_channels", "bandwidth")]


def build_hostsim(so=HOSTSIM_SO):
    subprocess.run(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-Wno-unused-function", "-o", so, HOSTSIM_SRC], check=True)


def _bind(lib, prefix):
    """The coding entry points shared by the host simulation (hostsim_*) and the reference harness (ref_*): same arguments."""
    getattr(lib, prefix + "decode_stream").argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                                       C.c_void_p, C.c_void_p, C.c_void_p]
    getattr(lib, prefix + "encode_stream").argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int,
                                                       C.c_void_p, C.c_void_p]
    getattr(lib, prefix + "encode_stream_script").argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                                              C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    return lib


_lib = None
_ref = None


def hostsim():
    """tests/hostsim/libhostsim.so (built by __graft_entry__.build(); built here when missing)."""
    global _lib
    if _lib is None:
        if not os.path.exists(HOSTSIM_SO):
            build_hostsim()
        lib = _bind(C.CDLL(HOSTSIM_SO), "hostsim_")
        lib.hostsim_generate_music.argtypes = [C.c_void_p, C.c_int32, C.c_uint32]
        _lib = lib
    return _lib


def _codec(name):
    """The oracle's entry point `name`: the reference build while recording digests, else the host simulation."""
    global _ref
    if not RECORD:
        return getattr(hostsim(), "hostsim_" + name)
    if _ref is None:
        if not os.path.exists(REF_SO):
            raise RuntimeError("ORACLE_DIGEST_RECORD records the reference's results: build oracle/_ref first "
                               "(make -C oracle REF=<opus-fix source tree>)")
        _ref = _bind(C.CDLL(REF_SO), "ref_")
    return getattr(_ref, "ref_" + name)


def ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


# ---- digests of the reference's results --------------------------------------------------------------------------------------

_table = None
_rec_lock = threading.Lock()


def _digest(*parts):
    h = hashlib.blake2b(digest_size=8)
    for p in parts:
        if isinstance(p, np.ndarray):
            p = np.ascontiguousarray(p)
            h.update(("%s%s" % (p.dtype.str, p.shape)).encode())
            h.update(p.tobytes())
        else:
            h.update(repr(p).encode())
        h.update(b"|")
    return int.from_bytes(h.digest(), "little")


def _stored():
    global _table
    if _table is None:
        t = np.load(DIGESTS) if os.path.exists(DIGESTS) else np.zeros((0, 2), dtype=np.uint64)
        _table = dict(zip(t[:, 0].tolist(), t[:, 1].tolist()))
    return _table


def _pin(kind, inputs, outputs):
    k, v = _digest(kind, *inputs), _digest(*outputs)
    if RECORD:
        with _rec_lock, open(RECORD, "a") as f:
            f.write("%016x %016x\n" % (k, v))
        return
    want = _stored().get(k)
    assert want is not None, ("oracle: no stored reference result for this %s call (new input?): record it from the reference build "
                              "(ORACLE_DIGEST_RECORD, see tests/oracle_lib.py), or pass pin=False where none is wanted" % kind)
    assert want == v, "oracle: the %s result differs from the reference's (tests/golden/oracle_digests.npy)" % kind


def _packets(out, stride, lens):
    """Bytes of the coded packets only (what follows a packet in its slot is not part of the result)."""
    rows = out.reshape(-1, stride)
    return np.concatenate([rows[f, :max(int(n), 0)] for f, n in enumerate(lens)] + [np.zeros(0, np.uint8)])


# ---- the oracle ---------------------------------------------------------------------------------------------------------------

def generate_music(n_samples, seed=13371337):
    """Stereo int16 [n_samples, 2] — the signal of opus-fix/tests/test_opus_encode.c:59-90."""
    buf = np.zeros((n_samples, 2), dtype=np.int16)
    hostsim().hostsim_generate_music(ptr(buf), n_samples, seed & 0xFFFFFFFF)
    return buf


def test_signal(n_samples, channels, seed=13371337, kind="music"):
    """Deterministic test signals: 'music' (generate_music), 'noise' (full-scale), 'tone' (pitched, drives the
    post-filter), 'clicks' (music + impulses, drives transients)."""
    rng = np.random.RandomState(seed & 0x7FFFFFFF)
    if kind == "music":
        x = generate_music(n_samples, seed)
    elif kind == "noise":
        x = rng.randint(-32768, 32768, size=(n_samples, 2)).astype(np.int16)
    elif kind == "tone":
        t = np.arange(n_samples)
        f0 = 180.0 + (seed % 7) * 37.0
        s = sum(np.sin(2 * np.pi * f0 * k * t / 48000.0) / k for k in range(1, 9))
        env = 0.6 + 0.4 * np.sin(2 * np.pi * t / 48000.0 * 0.7)
        y = (s * env * 6000).astype(np.int32)
        x = np.stack([y, (y * 0.8).astype(np.int32)], axis=1)
        x = (x + rng.randint(-40, 40, size=x.shape)).clip(-32768, 32767).astype(np.int16)
    elif kind == "clicks":
        x = generate_music(n_samples, seed).astype(np.int32) // 2
        pos = rng.randint(0, n_samples, size=max(1, n_samples // 9000))
        for p in pos:
            seg = x[p:p + 64]
            seg += (rng.randint(-20000, 20000, size=seg.shape))
        x = x.clip(-32768, 32767).astype(np.int16)
    else:
        raise ValueError(kind)
    if channels == 1:
        x = x[:, :1].copy()
    return np.ascontiguousarray(x)


def encode_stream(pcm, frame_size, bitrate, channels=None, Fs=48000, vbr=1, cvbr=0, complexity=10,
                  application=OPUS_APPLICATION_RESTRICTED_LOWDELAY, max_bytes=1275, stride=1276, force_channels=0, bandwidth=0,
                  pin=True):
    """Encode one stream.  Returns (data uint8 [F*stride], offs int64 [F], lens int32 [F], ranges uint32 [F]).
    A frame the reference codes with SILK / hybrid (OPUS_APPLICATION_AUDIO at low rates) is not CELT: its length is
    OPUS_UNIMPLEMENTED and the stream stops there (the TOC bytes of it and of every later frame read zero)."""
    pcm = np.ascontiguousarray(pcm, dtype=np.int16)
    if channels is None:
        channels = pcm.shape[1]
    F = pcm.shape[0] // frame_size
    out = np.zeros(F * stride, dtype=np.uint8)
    lens = np.zeros(F, dtype=np.int32)
    ranges = np.zeros(F, dtype=np.uint32)
    cfg = np.array([application, bitrate, vbr, cvbr, complexity, max_bytes, force_channels, bandwidth], dtype=np.int32)
    rc = _codec("encode_stream")(ptr(pcm), F, frame_size, channels, Fs, ptr(cfg), ptr(out), stride, ptr(lens), ptr(ranges))
    assert rc == 0 or rc == OPUS_UNIMPLEMENTED, rc
    if pin and rc == 0:   # a stream the reference codes partly with SILK has no result here to check
        _pin("encode", (pcm[:F * frame_size], frame_size, channels, Fs, cfg), (_packets(out, stride, lens), lens, ranges))
    offs = (np.arange(F, dtype=np.int64) * stride)
    return out, offs, lens, ranges


def pack(data, offs, lens):
    """Re-pack strided packets contiguously -> (data, offs[F])."""
    F = len(lens)
    noffs = np.zeros(F, dtype=np.int64)
    noffs[1:] = np.cumsum(lens[:-1].clip(min=0))
    total = int(noffs[-1] + max(int(lens[-1]), 0)) if F else 0
    out = np.zeros(max(total, 1), dtype=np.uint8)
    for f in range(F):
        n = int(lens[f])
        if n > 0:
            out[noffs[f]:noffs[f] + n] = data[offs[f]:offs[f] + n]
    return out, noffs


def decode_stream(data, offs, lens, frame_size, channels, Fs=48000, pin=True):
    """Decode one stream.  Returns (pcm int16 [F*frame_size, channels], ranges, rets)."""
    F = len(lens)
    offs = np.ascontiguousarray(offs, dtype=np.int64)
    lens = np.ascontiguousarray(lens, dtype=np.int32)
    pcm = np.zeros((F * frame_size, channels), dtype=np.int16)
    ranges = np.zeros(F, dtype=np.uint32)
    rets = np.zeros(F, dtype=np.int32)
    _codec("decode_stream")(ptr(data), ptr(offs), ptr(lens), F, frame_size, channels, Fs, ptr(pcm), ptr(ranges), ptr(rets))
    if pin:
        pk = np.concatenate([np.asarray(data[o:o + n], dtype=np.uint8) for o, n in zip(offs.tolist(), lens.tolist()) if n > 0]
                            + [np.zeros(0, np.uint8)])
        _pin("decode", (pk, lens, frame_size, channels, Fs), (pcm, ranges, rets))
    return pcm, ranges, rets


def _pool(n, threads, fn):
    """fn(i) for i < n on `threads` host threads (the oracle's calls release the GIL)."""
    nxt = [0]
    lock = threading.Lock()
    err = []

    def work():
        while not err:
            with lock:
                i = nxt[0]
                nxt[0] += 1
            if i >= n:
                return
            try:
                fn(i)
            except BaseException as e:   # re-raised below
                err.append(e)
    ths = [threading.Thread(target=work) for _ in range(max(1, min(threads, n)))]
    [t.start() for t in ths]
    [t.join() for t in ths]
    if err:
        raise err[0]


def encode_streams(pcm, frame_size, bitrate, threads, vbr=1, cvbr=0, complexity=10, Fs=48000, max_bytes=1276, stride=1276,
                   pin=True):
    """n independent streams pcm [n, T, channels], one per host thread at a time.
    Returns (packets uint8 [n, F, stride], lens int32 [n, F], ranges uint32 [n, F])."""
    n, T, ch = pcm.shape
    F = T // frame_size
    out = np.zeros((n, F, stride), dtype=np.uint8)
    lens = np.zeros((n, F), dtype=np.int32)
    ranges = np.zeros((n, F), dtype=np.uint32)

    def one(i):
        d, _, l, r = encode_stream(pcm[i], frame_size, bitrate, ch, Fs=Fs, vbr=vbr, cvbr=cvbr, complexity=complexity, max_bytes=max_bytes,
                                   stride=stride, pin=pin)
        out[i] = d.reshape(F, stride)
        lens[i] = l
        ranges[i] = r
    _pool(n, threads, one)
    return out, lens, ranges


def decode_streams(n, F, threads, data, offs, lens, frame_size, channels, Fs=48000, pin=True):
    """n independent streams of F packets each (stream s owns packets s*F .. s*F+F-1 of the packed layout), one per host
    thread at a time.  Returns (pcm int16 [n*F*frame_size, channels], ranges uint32 [n*F], rets int32 [n*F])."""
    pcm = np.zeros((n * F * frame_size, channels), dtype=np.int16)
    ranges = np.zeros(n * F, dtype=np.uint32)
    rets = np.zeros(n * F, dtype=np.int32)

    def one(s):
        sl = slice(s * F, (s + 1) * F)
        p, r, t = decode_stream(data, offs[sl], lens[sl], frame_size, channels, Fs=Fs, pin=False)
        pcm[s * F * frame_size:(s + 1) * F * frame_size] = p
        ranges[sl] = r
        rets[sl] = t
    _pool(n, threads, one)
    if pin:
        pk = np.concatenate([np.asarray(data[o:o + m], dtype=np.uint8) for o, m in zip(offs.tolist(), lens.tolist()) if m > 0]
                            + [np.zeros(0, np.uint8)])
        _pin("decode_streams", (pk, np.ascontiguousarray(lens, dtype=np.int32), n, F, frame_size, channels, Fs), (pcm, ranges, rets))
    return pcm, ranges, rets


def ctl_script(seed, F, channels, K=2, allow_mode=False):
    """Random encoder ctl changes, K slots before every frame: int32 [F, K, 2] of (request, value); request 0 = nothing.
    The shape of the reference's own encoder fuzz loop (opus-fix/tests/test_opus_encode.c:236-330)."""
    rs = np.random.RandomState(seed)
    script = np.zeros((F, K, 2), dtype=np.int32)
    for f in range(F):
        for k in range(K):
            if rs.rand() >= 0.25:
                continue
            c = rs.randint(12)
            if c == 0:
                script[f, k] = (4002, int(rs.choice([6000, 12000, 24000, 32000, 48000, 64000, 96000, 128000, 256000, 510000, -1000, -1])))
            elif c == 1:
                script[f, k] = (4006, rs.randint(2))
            elif c == 2:
                script[f, k] = (4020, rs.randint(2))
            elif c == 3:
                script[f, k] = (4010, rs.randint(11))
            elif c == 4:
                script[f, k] = (4022, int(rs.choice([1, 2, -1000])) if channels == 2 else -1000)
            elif c == 5:
                script[f, k] = (4008, int(rs.choice([-1000, 1101, 1102, 1103, 1104, 1105])))
            elif c == 6:
                script[f, k] = (4004, int(rs.choice([1101, 1102, 1103, 1104, 1105])))
            elif c == 7:
                script[f, k] = (4014, rs.randint(0, 30))
            elif c == 8:
                script[f, k] = (4036, rs.randint(8, 25))
            elif c == 9:
                script[f, k] = (4042, rs.randint(2))
            elif c == 10:
                script[f, k] = (4024, int(rs.choice([-1000, 3001, 3002])))
            elif rs.rand() < 0.2:
                script[f, k] = (4028, 0)
    return script


def encode_stream_script(pcm, frame_size, channels, script, Fs=48000, application=OPUS_APPLICATION_RESTRICTED_LOWDELAY, stride=1276,
                         pin=True):
    """Encode with a ctl script.  Returns (packets [F, stride], lens, ranges)."""
    pcm = np.ascontiguousarray(pcm, dtype=np.int16)
    script = np.ascontiguousarray(script, dtype=np.int32)
    F, K = script.shape[0], script.shape[1]
    out = np.zeros((F, stride), dtype=np.uint8)
    lens = np.zeros(F, dtype=np.int32)
    ranges = np.zeros(F, dtype=np.uint32)
    cfg = np.array([application, 64000, 1, 1, 10, stride, 0, 0], dtype=np.int32)
    _codec("encode_stream_script")(ptr(pcm), F, frame_size, channels, Fs, ptr(cfg), ptr(script), K, ptr(out), stride, ptr(lens),
                                   ptr(ranges))
    if pin:
        _pin("encode_script", (pcm[:F * frame_size], frame_size, channels, Fs, cfg, script),
             (_packets(out, stride, lens), lens, ranges))
    return out, lens, ranges


def record(path):
    """Merge the lines an ORACLE_DIGEST_RECORD run (the oracle on the reference build) appended to `path` into
    tests/golden/oracle_digests.npy."""
    rows = {}
    for t in (np.load(DIGESTS) if os.path.exists(DIGESTS) else np.zeros((0, 2), dtype=np.uint64)).tolist():
        rows[t[0]] = t[1]
    for line in open(path):
        k, v = (int(x, 16) for x in line.split())
        assert rows.get(k, v) == v, "conflicting digests for one call"
        rows[k] = v
    keys = sorted(rows)
    np.save(DIGESTS, np.array([[k, rows[k]] for k in keys], dtype=np.uint64).reshape(-1, 2))
    print("%d digests in %s" % (len(keys), DIGESTS))


if __name__ == "__main__":
    if len(sys.argv) == 3 and sys.argv[1] == "record":
        record(sys.argv[2])
    else:
        raise SystemExit("usage: python tests/oracle_lib.py record DIGEST_LINES")

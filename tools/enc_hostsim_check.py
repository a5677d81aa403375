"""Dev tool: compare the host simulation of the encoder (tests/hostsim) with the oracle, packet by packet."""
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import oracle_lib as O

H = C.CDLL(os.path.join(ROOT, "tests", "hostsim", "libhostsim.so"))
H.hostsim_encode_stream.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]


def sim_encode(pcm, frame_size, bitrate, channels, vbr=1, cvbr=0, complexity=10, application=O.OPUS_APPLICATION_RESTRICTED_LOWDELAY,
               max_bytes=1275, stride=1276, force_channels=0, bandwidth=0):
    pcm = np.ascontiguousarray(pcm, dtype=np.int16)
    F = pcm.shape[0] // frame_size
    out = np.zeros(F * stride, dtype=np.uint8)
    lens = np.zeros(F, dtype=np.int32)
    ranges = np.zeros(F, dtype=np.uint32)
    cfg = np.array([application, bitrate, vbr, cvbr, complexity, max_bytes, force_channels, bandwidth], dtype=np.int32)
    rc = H.hostsim_encode_stream(O.ptr(pcm), F, frame_size, channels, 48000, O.ptr(cfg), O.ptr(out), stride, O.ptr(lens), O.ptr(ranges))
    return out, lens, ranges, rc


def compare(kind, channels, frame_size, bitrate, vbr, cvbr, complexity, seconds=2, seed=1234, verbose=True):
    pcm = O.test_signal(48000 * seconds, channels, seed, kind)
    d, o, l, r = O.encode_stream(pcm, frame_size, bitrate, channels, vbr=vbr, cvbr=cvbr, complexity=complexity, pin=False)
    d2, l2, r2, rc = sim_encode(pcm, frame_size, bitrate, channels, vbr=vbr, cvbr=cvbr, complexity=complexity)
    F = len(l)
    bad = -1
    for f in range(F):
        if l[f] != l2[f] or r[f] != r2[f] or not np.array_equal(d[o[f]:o[f] + l[f]], d2[f * 1276:f * 1276 + l[f]]):
            bad = f
            break
    tag = "%s ch%d fs%d br%d vbr%d cvbr%d cx%d" % (kind, channels, frame_size, bitrate, vbr, cvbr, complexity)
    if bad < 0:
        if verbose:
            print("OK   ", tag, "frames", F, "mean bytes %.1f" % l.mean())
        return True
    a = d[o[bad]:o[bad] + l[bad]]
    b = d2[bad * 1276:bad * 1276 + max(l2[bad], 0)]
    n = min(len(a), len(b))
    diff = np.nonzero(a[:n] != b[:n])[0]
    print("FAIL ", tag, "first bad frame", bad, "of", F, "len ref/sim", l[bad], l2[bad], "rng %08x/%08x" % (r[bad], r2[bad]),
          "first diff byte", (diff[0] if len(diff) else n), "rc", rc)
    return False


if __name__ == "__main__":
    ok = True
    quick = [("music", 2, 960, 64000, 0, 0, 10), ("music", 2, 960, 96000, 1, 0, 10), ("music", 1, 960, 64000, 1, 1, 10),
             ("tone", 2, 960, 96000, 1, 0, 10), ("clicks", 2, 960, 96000, 1, 0, 10), ("noise", 2, 960, 128000, 1, 0, 10)]
    for q in quick:
        ok &= compare(*q)
    sys.exit(0 if ok else 1)

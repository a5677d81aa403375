#!/usr/bin/env python
"""ms_bench.py — multistream decode throughput on one GPU: a 5.1 layout (streams=4, coupled=2, mapping [0,4,1,2,3,5]: two stereo
and two mono streams per decoder), --n multistream decoders, --frames frames of 20 ms, inputs and outputs resident on the device.

  (a) opus_multistream_decode_span_device over the multistream packets
  (b) the same elementary packets through opus_decode_span_device as two uniform-channel calls (the stereo and the mono streams)

(a) and (b) run alternately in one process; each repeat times one call of each (host clock around the call and
opus_b200_synchronize).  Reports x realtime per multistream stream (audio seconds of one 5.1 stream per wall second), the spread
over the repeats, the device time of the split and gather stages of (a) (CUDA events), and the card's name and power limit.
Inputs come from the library's encoder (stereo 128 kbps and mono 64 kbps VBR, complexity 10).  Writes DIR/ms_bench.json."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import concentus_b200 as cb  # noqa: E402
import ms_framing as M  # noqa: E402
import oracle_lib as O  # noqa: E402

MAPPING = [0, 4, 1, 2, 3, 5]
S, COUPLED, CH, FS = 4, 2, 6, 960


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=60).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as e:   # no nvidia-smi: the name from CUDA, no power limit
        import torch
        return "%s, power limit unknown (%s)" % (torch.cuda.get_device_name(0), type(e).__name__)


def encode(n, channels, bitrate, frames, seed):
    """n streams of `frames` 20 ms packets from the library's encoder -> list of lists of bytes."""
    srcs = [O.test_signal(FS * frames, channels, seed + k, "music") for k in range(16)]
    pcm = np.stack([np.roll(srcs[i % 16], 4801 * (i // 16), axis=0) for i in range(n)])
    enc = cb.EncoderBatch(n, 48000, channels, application=cb.OPUS_APPLICATION_RESTRICTED_LOWDELAY, bitrate=bitrate, vbr=1, cvbr=0,
                          complexity=10)
    data, lens = enc.encode_span(pcm.reshape(-1, channels), frames, FS)
    enc.close()
    assert (lens > 0).all()
    return [[bytes(data[i * frames + f, :lens[i * frames + f]]) for f in range(frames)] for i in range(n)]


def self_delimit_code0(p):
    assert p[0] & 3 == 0
    return p[:1] + M.size_bytes(len(p) - 1) + p[1:]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1024, help="multistream decoders")
    ap.add_argument("--frames", type=int, default=300)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default="ms_bench_out", help="directory for ms_bench.json")
    a = ap.parse_args()
    import torch
    L = cb.lib()
    assert L.opus_b200_init(0) == 0, "no CUDA device"
    dev = torch.device("cuda", 0)
    n, F = a.n, a.frames
    name = card()
    print("card:", name, flush=True)
    t0 = time.time()
    st = encode(2 * n, 2, 128000, F, 100)
    mo = encode(2 * n, 1, 64000, F, 200)
    # multistream decoder m: stereo streams 2m, 2m+1 and mono streams 2m, 2m+1
    ms = [self_delimit_code0(st[2 * m][f]) + self_delimit_code0(st[2 * m + 1][f]) + self_delimit_code0(mo[2 * m][f]) + mo[2 * m + 1][f]
          for m in range(n) for f in range(F)]
    blob, offs, lens = M.ms_blob(ms)
    sb, so, sl = M.ms_blob([p for s in st for p in s])
    mb, mo_, ml = M.ms_blob([p for s in mo for p in s])
    print("inputs: %.1f s, %.1f MB multistream packets" % (time.time() - t0, blob.nbytes / 1e6), flush=True)
    T = lambda x: torch.from_numpy(x).to(dev)   # noqa: E731
    d_ms = [T(blob), T(offs), T(lens)]
    d_st = [T(sb), T(so), T(sl)]
    d_mo = [T(mb), T(mo_), T(ml)]
    d_pcm_a = torch.empty((n * F * FS * CH,), dtype=torch.int16, device=dev)
    d_ret_a = torch.empty((n * F,), dtype=torch.int32, device=dev)
    d_pcm_s = torch.empty((2 * n * F * FS * 2,), dtype=torch.int16, device=dev)
    d_ret_s = torch.empty((2 * n * F,), dtype=torch.int32, device=dev)
    d_pcm_m = torch.empty((2 * n * F * FS,), dtype=torch.int16, device=dev)
    d_ret_m = torch.empty((2 * n * F,), dtype=torch.int32, device=dev)
    msd = cb.MSDecoderBatch(n, 48000, CH, S, COUPLED, MAPPING)
    sd = cb.DecoderBatch(2 * n, 48000, 2)
    md = cb.DecoderBatch(2 * n, 48000, 1)
    P = lambda t: C.c_void_p(t.data_ptr())   # noqa: E731

    def run_a():
        rc = L.opus_multistream_decode_span_device(msd.handles, n, F, P(d_ms[0]), P(d_ms[1]), P(d_ms[2]), P(d_pcm_a), FS, P(d_ret_a))
        assert rc == 0 and L.opus_b200_synchronize() == 0

    def run_b():
        rc = L.opus_decode_span_device(sd.handles, 2 * n, F, P(d_st[0]), P(d_st[1]), P(d_st[2]), P(d_pcm_s), FS, P(d_ret_s))
        rc2 = L.opus_decode_span_device(md.handles, 2 * n, F, P(d_mo[0]), P(d_mo[1]), P(d_mo[2]), P(d_pcm_m), FS, P(d_ret_m))
        assert rc == 0 and rc2 == 0 and L.opus_b200_synchronize() == 0

    # warm-up pass from fresh states: (a) must equal (b) with the mapping applied
    run_a()
    run_b()
    assert bool((d_ret_a == FS).all()) and bool((d_ret_s == FS).all()) and bool((d_ret_m == FS).all())
    for m in (0, n // 3, n - 1):
        a_ = d_pcm_a.view(n, F, FS, CH)[m]
        s_ = d_pcm_s.view(2 * n, F, FS, 2)
        m_ = d_pcm_m.view(2 * n, F, FS)
        # output channels [0,4,1,2,3,5] of stream channels: L0, mono stream 2, R0, L1, R1, mono stream 3
        want = torch.stack([s_[2 * m, :, :, 0], m_[2 * m], s_[2 * m, :, :, 1], s_[2 * m + 1, :, :, 0], s_[2 * m + 1, :, :, 1],
                            m_[2 * m + 1]], dim=-1)
        assert torch.equal(a_, want), "multistream output differs from the single-stream decoders (decoder %d)" % m
    audio = F * FS / 48000.0   # seconds of one stream
    ta, tb, split, gather = [], [], [], []
    ms2 = (C.c_double * 2)()
    ln2 = (C.c_longlong * 2)()
    for r in range(a.repeats):
        L.opus_b200_ms_stage_times(ms2, ln2, 1)
        t = time.perf_counter()
        run_a()
        ta.append(time.perf_counter() - t)
        L.opus_b200_ms_stage_times(ms2, ln2, 1)
        split.append(ms2[0])
        gather.append(ms2[1])
        t = time.perf_counter()
        run_b()
        tb.append(time.perf_counter() - t)
        print("repeat %d: (a) %.1f ms  (b) %.1f ms  split %.2f ms  gather %.2f ms" % (r, ta[-1] * 1e3, tb[-1] * 1e3, split[-1], gather[-1]),
              flush=True)
    xa = [n * audio / t for t in ta]
    xb = [n * audio / t for t in tb]
    res = {
        "card": name,
        "workload": "5.1 (streams=4, coupled=2, mapping %s), %d multistream decoders = %d stereo + %d mono elementary, %d x 20 ms, "
                    "device-resident, library encoder 128 kbps stereo / 64 kbps mono VBR" % (MAPPING, n, 2 * n, 2 * n, F),
        "a_multistream_span_device_xrt": {"median": float(np.median(xa)), "min": float(min(xa)), "max": float(max(xa))},
        "b_two_uniform_span_device_xrt": {"median": float(np.median(xb)), "min": float(min(xb)), "max": float(max(xb))},
        "a_ms": [t * 1e3 for t in ta], "b_ms": [t * 1e3 for t in tb],
        "split_ms": split, "gather_ms": gather,
        "split_gather_share_of_a": float(np.median([(s + g) / (t * 1e3) for s, g, t in zip(split, gather, ta)])),
    }
    print(json.dumps(res, indent=1))
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "ms_bench.json"), "w") as f:
        json.dump(res, f, indent=1)
    for d in (msd, sd, md):
        d.close()


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""synth_stage_bench.py — device time of each decoder pipeline stage (parse, synth, de-emphasis) on one GPU, one chunk per call.

--streams stereo decoders (default 4,096, the headline's batch) decode --frames 20 ms packets per call (default 108, one pipeline
chunk of the headline), inputs and outputs resident on the device.  A call of a single chunk runs its three stages one after another,
so each stage's CUDA-event time is its time alone, not time shared with the next chunk's parse.  Packets are 64 kbps CBR from the
library's encoder (restricted low delay, complexity 10), the headline's setting; every call decodes the same packets, the decoders'
state carrying on from call to call.

Reports ms per launch of every stage over --calls timed calls after --warmup calls, the wall time of a call (host clock around the
call and opus_b200_synchronize), and the card's name and power limit read in the same run.  Writes DIR/synth_stage_bench.json.
Compare library builds by running it once per build (CB200_LIB=<path>.so), alternating."""
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
import oracle_lib as O  # noqa: E402

FS, CH = 960, 2
STAGES = ["parse_kernel", "synth_kernel", "deemph_kernel"]


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=60).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as e:   # no nvidia-smi: the name from CUDA, no power limit
        import torch
        return "%s, power limit unknown (%s)" % (torch.cuda.get_device_name(0), type(e).__name__)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=4096)
    ap.add_argument("--frames", type=int, default=108, help="packets per stream and call (one pipeline chunk)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--out", default="synth_stage_bench_out", help="directory for synth_stage_bench.json")
    a = ap.parse_args()
    import torch
    L = cb.lib()
    assert L.opus_b200_init(0) == 0, "no CUDA device"
    dev = torch.device("cuda", 0)
    n, F = a.streams, a.frames
    name = card()
    print("card:", name, "library:", cb.LIB_PATH, flush=True)

    # inputs: 16 distinct signals, each stream a rotated copy of one of them
    srcs = [O.test_signal(FS * F, CH, 300 + k, "music" if k % 4 else "tone") for k in range(16)]
    pcm = np.stack([np.roll(srcs[i % 16], 4801 * (i // 16), axis=0) for i in range(n)])
    enc = cb.EncoderBatch(n, 48000, CH, application=cb.OPUS_APPLICATION_RESTRICTED_LOWDELAY, bitrate=64000, vbr=0, cvbr=0, complexity=10)
    data, lens = enc.encode_span(pcm.reshape(-1, CH), F, FS)
    enc.close()
    del pcm
    lens = lens.astype(np.int32)
    assert (lens > 0).all()
    stride = data.shape[1]
    offs = (np.arange(n * F, dtype=np.int64) * stride)
    d_data = torch.from_numpy(np.ascontiguousarray(data).reshape(-1)).to(dev)
    d_offs = torch.from_numpy(offs).to(dev)
    d_lens = torch.from_numpy(lens.reshape(-1)).to(dev)
    d_pcm = torch.empty((n * F * FS * CH,), dtype=torch.int16, device=dev)
    d_ret = torch.empty((n * F,), dtype=torch.int32, device=dev)
    dec = cb.DecoderBatch(n, 48000, CH)
    P = lambda t: C.c_void_p(t.data_ptr())   # noqa: E731

    def call():
        rc = L.opus_decode_span_device(dec.handles, n, F, P(d_data), P(d_offs), P(d_lens), P(d_pcm), FS, P(d_ret))
        assert rc == 0 and L.opus_b200_synchronize() == 0

    for _ in range(a.warmup):
        call()
    assert bool((d_ret == FS).all()), "decode returned errors"
    ms = (C.c_double * 3)()
    nl = (C.c_longlong * 3)()
    L.opus_b200_stage_times(None, None, 1)
    wall = []
    for _ in range(a.calls):
        t = time.perf_counter()
        call()
        wall.append((time.perf_counter() - t) * 1e3)
    L.opus_b200_stage_times(ms, nl, 0)
    assert bool((d_ret == FS).all()), "decode returned errors"
    stages = {}
    for i, nm in enumerate(STAGES):
        assert nl[i] == a.calls, "%s: %d launches in %d calls (expected one chunk per call)" % (nm, nl[i], a.calls)
        stages[nm] = {"launches": int(nl[i]), "ms_per_launch": ms[i] / nl[i]}
    res = {
        "card": name,
        "library": os.path.basename(cb.LIB_PATH),
        "workload": "%d stereo decoders x %d x 20 ms per call (one chunk), 64 kbps CBR, device-resident; %d warm-up + %d timed calls"
                    % (n, F, a.warmup, a.calls),
        "stages": stages,
        "call_ms": {"median": float(np.median(wall)), "min": float(min(wall)), "max": float(max(wall))},
    }
    print(json.dumps(res, indent=1))
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "synth_stage_bench.json"), "w") as f:
        json.dump(res, f, indent=1)
    dec.close()


if __name__ == "__main__":
    main()

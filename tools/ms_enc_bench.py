#!/usr/bin/env python
"""ms_enc_bench.py — multistream encode throughput on one GPU: a 5.1 layout (streams=4, coupled=2, mapping [0,4,1,2,3,5]: two
stereo and two mono streams per encoder), --n multistream encoders, --frames frames of 20 ms, 256 kbps VBR, complexity 10,
max_data_bytes 6144, inputs and outputs resident on the device.

  (a) opus_multistream_encode_span_device (the merged schedule)
  (b) the same elementary streams through opus_encode_span_device as two uniform-channel calls at the bitrates the multistream
      encoder allocates (78,666 b/s per stereo stream, 49,333 b/s per mono stream); its packets are framed afterwards (for the
      check only).  (a) and (b) must be byte-identical: checked on the first repeat, from fresh states, for a sample of encoders.
  (c) the layout of (a) in CBR (the ordered schedule: one pass per stream), for the record.

(a), (b) and (c) run alternately in one process; each repeat times one call of each (host clock around the call and
opus_b200_enc_synchronize).  Reports x realtime per multistream stream (audio seconds of one 5.1 stream per wall second), the spread
over the repeats, the device time of the route / budget / pack kernels (CUDA events), and the card's name and power limit.
Input: 16 seeded 6-channel signals, each encoder's a distinct rotation of one of them.  Writes DIR/ms_enc_bench_<n>.json."""
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
import ms_enc_framing as E  # noqa: E402
import oracle_lib as O  # noqa: E402

MAPPING = [0, 4, 1, 2, 3, 5]
S, COUPLED, CH, FS, BITRATE, MAXB = 4, 2, 6, 960, 256000, 6144


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
    ap.add_argument("--n", type=int, nargs="+", default=[1024, 2048], help="multistream encoders")
    ap.add_argument("--frames", type=int, default=300)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--check", type=int, default=8, help="encoders whose (a) and (b) packets are compared")
    ap.add_argument("--out", default="ms_enc_bench_out", help="directory for the JSON results")
    a = ap.parse_args()
    import torch
    L = cb.lib()
    assert L.opus_b200_init(0) == 0, "no CUDA device"
    dev = torch.device("cuda", 0)
    name = card()
    print("card:", name, flush=True)
    F, T = a.frames, a.frames * FS
    rates = E.ms_rates(BITRATE, CH, S, COUPLED, 48000, FS)
    assert rates == [78666, 78666, 49333, 49333], rates
    base = torch.from_numpy(np.stack([np.concatenate([O.test_signal(T, 2, 1000 + 3 * k + j, ("music", "tone", "clicks")[j])
                                                      for j in range(3)], axis=1) for k in range(16)])).to(dev)
    P = lambda t: C.c_void_p(t.data_ptr())   # noqa: E731
    os.makedirs(a.out, exist_ok=True)
    for n in a.n:
        pcm = torch.empty((n, T, CH), dtype=torch.int16, device=dev)
        for i in range(n):
            pcm[i] = torch.roll(base[i % 16], shifts=4801 * (i // 16) + 97 * (i % 16), dims=0)
        # (b)'s inputs: stream channel k <- input channel MAPPING.index(k)
        src = [MAPPING.index(k) for k in range(S + COUPLED)]
        st_pcm = torch.stack([pcm[:, :, [src[0], src[1]]], pcm[:, :, [src[2], src[3]]]], dim=1).contiguous()   # [n, 2, T, 2]
        mo_pcm = torch.stack([pcm[:, :, src[4]], pcm[:, :, src[5]]], dim=1).contiguous()                     # [n, 2, T]
        d_a = torch.empty((n * F * MAXB,), dtype=torch.uint8, device=dev)
        r_a = torch.empty((n * F,), dtype=torch.int32, device=dev)
        d_c = torch.empty((n * F * MAXB,), dtype=torch.uint8, device=dev)
        r_c = torch.empty((n * F,), dtype=torch.int32, device=dev)
        d_s = torch.empty((2 * n * F * 1276,), dtype=torch.uint8, device=dev)
        r_s = torch.empty((2 * n * F,), dtype=torch.int32, device=dev)
        d_m = torch.empty((2 * n * F * 1276,), dtype=torch.uint8, device=dev)
        r_m = torch.empty((2 * n * F,), dtype=torch.int32, device=dev)
        torch.cuda.synchronize()
        msa = cb.MSEncoderBatch(n, 48000, CH, S, COUPLED, MAPPING, bitrate=BITRATE, vbr=1, cvbr=0, complexity=10)
        msc = cb.MSEncoderBatch(n, 48000, CH, S, COUPLED, MAPPING, bitrate=BITRATE, vbr=0, cvbr=0, complexity=10)
        se = cb.EncoderBatch(2 * n, 48000, 2, bitrate=rates[0], vbr=1, cvbr=0, complexity=10)
        me = cb.EncoderBatch(2 * n, 48000, 1, bitrate=rates[2], vbr=1, cvbr=0, complexity=10)

        def run_a():
            assert L.opus_multistream_encode_span_device(msa.handles, n, F, P(pcm), FS, P(d_a), MAXB, P(r_a)) == 0
            assert L.opus_b200_enc_synchronize() == 0

        def run_b():
            assert L.opus_encode_span_device(se.handles, 2 * n, F, P(st_pcm), FS, P(d_s), 1276, P(r_s)) == 0
            assert L.opus_encode_span_device(me.handles, 2 * n, F, P(mo_pcm), FS, P(d_m), 1276, P(r_m)) == 0
            assert L.opus_b200_enc_synchronize() == 0

        def run_c():
            assert L.opus_multistream_encode_span_device(msc.handles, n, F, P(pcm), FS, P(d_c), MAXB, P(r_c)) == 0
            assert L.opus_b200_enc_synchronize() == 0

        audio = F * FS / 48000.0   # seconds of one stream
        res = {"card": name, "n": n,
               "workload": "5.1 (streams=4, coupled=2, mapping %s), %d multistream encoders = %d stereo + %d mono elementary, %d x 20 ms, "
                           "256 kbps VBR complexity 10, max_data_bytes %d, device-resident" % (MAPPING, n, 2 * n, 2 * n, F, MAXB)}
        times = {"a": [], "b": [], "c": []}
        stages = {"a": [], "c": []}
        ms3 = (C.c_double * 3)()
        ln3 = (C.c_longlong * 3)()
        for r in range(a.repeats + 1):   # repeat 0 is the warm-up (and the check, from fresh states)
            for k, fn in (("a", run_a), ("b", run_b), ("c", run_c)):
                L.opus_b200_ms_enc_stage_times(ms3, ln3, 1)
                t = time.perf_counter()
                fn()
                dt = time.perf_counter() - t
                L.opus_b200_ms_enc_stage_times(ms3, ln3, 1)
                if r > 0:
                    times[k].append(dt)
                    if k in stages:
                        stages[k].append({"route_ms": ms3[0], "budget_ms": ms3[1], "pack_ms": ms3[2]})
            if r == 0:
                assert bool((r_a > 0).all()) and bool((r_c > 0).all()) and bool((r_s > 0).all()) and bool((r_m > 0).all())
                A = d_a.view(n, F, MAXB)
                RA = r_a.view(n, F).cpu().numpy()
                BS, RS = d_s.view(2 * n, F, 1276), r_s.view(2 * n, F).cpu().numpy()
                BM, RM = d_m.view(2 * n, F, 1276), r_m.view(2 * n, F).cpu().numpy()
                for m in np.linspace(0, n - 1, a.check).astype(int):
                    Am, Bs0, Bs1, Bm0, Bm1 = (t[i].cpu().numpy() for t, i in ((A, m), (BS, 2 * m), (BS, 2 * m + 1), (BM, 2 * m), (BM, 2 * m + 1)))
                    for f in range(F):
                        subs = [bytes(Bs0[f, :RS[2 * m, f]]), bytes(Bs1[f, :RS[2 * m + 1, f]]), bytes(Bm0[f, :RM[2 * m, f]]),
                                bytes(Bm1[f, :RM[2 * m + 1, f]])]
                        want = b"".join(E.ms_frame(p, s < S - 1) for s, p in enumerate(subs))
                        assert RA[m, f] == len(want) and bytes(Am[f, :RA[m, f]]) == want, \
                            "(a) differs from the framed packets of (b): encoder %d frame %d" % (m, f)
                print("n=%d: (a) == framed (b) for %d encoders x %d frames" % (n, a.check, F), flush=True)
            else:
                print("n=%d repeat %d: (a) %.1f ms  (b) %.1f ms  (c) %.1f ms  (a) route %.2f pack %.2f  (c) route %.2f budget %.2f pack %.2f ms"
                      % (n, r, times["a"][-1] * 1e3, times["b"][-1] * 1e3, times["c"][-1] * 1e3, stages["a"][-1]["route_ms"],
                         stages["a"][-1]["pack_ms"], stages["c"][-1]["route_ms"], stages["c"][-1]["budget_ms"], stages["c"][-1]["pack_ms"]),
                      flush=True)
        for k, label in (("a", "a_multistream_span_device_merged_xrt"), ("b", "b_two_uniform_span_device_xrt"),
                         ("c", "c_multistream_span_device_cbr_ordered_xrt")):
            x = [n * audio / t for t in times[k]]
            res[label] = {"median": float(np.median(x)), "min": float(min(x)), "max": float(max(x))}
            res[k + "_ms"] = [t * 1e3 for t in times[k]]
        res["a_stages"], res["c_stages"] = stages["a"], stages["c"]
        print(json.dumps(res, indent=1), flush=True)
        with open(os.path.join(a.out, "ms_enc_bench_%d.json" % n), "w") as f:
            json.dump(res, f, indent=1)
        for b in (msa, msc, se, me):
            b.close()
        del pcm, st_pcm, mo_pcm, d_a, d_c, d_s, d_m
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()

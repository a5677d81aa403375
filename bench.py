#!/usr/bin/env python
"""bench.py — CELT decode (headline) and encode throughput (audio-seconds per wall-second, x realtime) on N B200s.

Workloads (BASELINE.json `configs`):
  [1] decode   4,096 independent 48 kHz stereo 64 kbps (CBR) 20 ms CELT streams, 60 s each, per GPU  -> the headline line
  [2] encode   4,096 streams, 48 kHz stereo, 96 kbps VBR, complexity 10                                -> the "encode" object
  [4] mixed    65,536 streams in total (sharded over the GPUs), per-stream bitrate drawn (seeded) from the sweep set
               32..510 kbps, CBR / VBR mix, decode + encode                                          -> the "mixed" object
One "step" = one pass over the whole batch.  Streams are sharded across GPUs by host-side partitioning (concentus_b200/shard.py),
no collective on the data path; [1] and [2] are weak scaling (per-GPU work fixed), [4] is strong scaling (total fixed).

Arms
  default            our CUDA engine through the C ABI of libconcentus_b200.so
                       value : packets and PCM resident in HBM (opus_decode_span_device / opus_encode_span_device)
                       e2e   : pinned host buffers in and out through opus_decode_span / opus_encode_span (H2D + D2H inside the timing)
  --impl reference   the UNMODIFIED opus-fix C build (oracle/_ref, built by `make -C oracle REF=<opus-fix source tree>`), one
                     stream per thread on all host cores, on a bounded sample of the same workload.  The same build gives the
                     "cpu_baseline" objects of the default arm; without it they are null.

Signals (BASELINE.md section 3): stream s plays generate_music with seed 13371337 + s (opus-fix/tests/test_opus_encode.c:59-90);
every eighth stream instead plays the reference's own parity input `48Khz Stereo.raw` (tests/golden/48Khz_Stereo.raw), cyclically
shifted by a per-stream offset.  Every stream has `--unique` seconds of its own signal, repeated to the workload's length (the decode
input is the oracle's encoding of those seconds, its packets repeated: the decoder sees a splice every `--unique` seconds, which is
as valid a packet sequence as any).  Clicks are added to a quarter of the music streams so that transients / short MDCTs occur.
The oracle is tests/oracle_lib.py.  The reference's results are stored only for the test suite's inputs, so here the oracle is the
host simulation of the codec headers, unchecked (pin=False): the parity passes compare the CUDA build with a host build of the same
headers, and the decode input is coded by the build's own encoder headers.  The result line carries a digest of each decode
workload's packets ("input_digest"), so runs of two builds can confirm that they decoded the same input.

--dump-outputs DIR writes, after the timed steps, what the timed calls of each workload returned in their last step (PCM and
return codes of the decode calls, packets and lengths of the encode calls) as DIR/<name>.npy: a fixed, seeded sample of 32 streams
x 50 frames per workload (float32, plus float64 indices of the sample; at most 42 MB in all, whatever the workload's size), so that
two builds can be compared output for output.
"""
import argparse
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

FS = 48000
CH = 2
FRAME = 960
BITRATE = 64000
ENC_BITRATE = 96000
SWEEP_RATES = [32000, 48000, 64000, 96000, 128000, 192000, 256000, 510000]
METRIC = "CELT decode audio-sec per sec (x realtime), 48k stereo"
ENC_METRIC = "CELT encode audio-sec per sec (x realtime), 48k stereo"
RAW_FIXTURE = os.path.join(ROOT, "tests", "golden", "48Khz_Stereo.raw")


# ------------------------------------------------------------------------------------------------------------------------------
# signals
# ------------------------------------------------------------------------------------------------------------------------------
def stream_signals(first, count, seconds, threads):
    """PCM of streams first .. first+count-1: int16 [count, seconds*FS, CH]."""
    import oracle_lib as O
    n_s = seconds * FS
    out = np.zeros((count, n_s, CH), dtype=np.int16)
    raw = np.fromfile(RAW_FIXTURE, dtype="<i2").reshape(-1, CH) if os.path.exists(RAW_FIXTURE) else None

    def work(k):
        s = first + k
        if raw is not None and s % 8 == 7:
            shift = (s * 7919) % (raw.shape[0] - n_s) if raw.shape[0] > n_s else 0
            seg = raw[shift:shift + n_s]
            out[k, :len(seg)] = seg
            if len(seg) < n_s:
                out[k, len(seg):] = np.resize(seg, (n_s - len(seg), CH))
        else:
            out[k] = O.generate_music(n_s, (13371337 + s) & 0xFFFFFFFF)
            if s % 4 == 1:   # clicks: drive the transient detector / short blocks / anti-collapse
                rs = np.random.RandomState(s)
                x = out[k].astype(np.int32) // 2
                for p in rs.randint(0, n_s - 64, size=max(1, n_s // 9000)):
                    x[p:p + 64] += rs.randint(-20000, 20000, size=(64, CH))
                out[k] = x.clip(-32768, 32767).astype(np.int16)

    ths = [threading.Thread(target=lambda lo=lo: [work(k) for k in range(lo, count, threads)]) for lo in range(threads)]
    [t.start() for t in ths]
    [t.join() for t in ths]
    return out


def oracle_encode(pcm, bitrates, vbr, cvbr, threads, stride):
    """Encode [n, T, CH] with the oracle (restricted-lowdelay, complexity 10), per-stream settings allowed.
    Returns (packets uint8 [n, F, stride], lens int32 [n, F])."""
    import oracle_lib as O
    n = pcm.shape[0]
    F = pcm.shape[1] // FRAME
    out = np.zeros((n, F, stride), dtype=np.uint8)
    lens = np.zeros((n, F), dtype=np.int32)
    bitrates = np.broadcast_to(np.asarray(bitrates), (n,))
    vbr = np.broadcast_to(np.asarray(vbr), (n,))
    cvbr = np.broadcast_to(np.asarray(cvbr), (n,))
    keys = sorted(set(zip(bitrates.tolist(), vbr.tolist(), cvbr.tolist())))
    for (br, v, cv) in keys:   # one setting per call
        idx = np.nonzero((bitrates == br) & (vbr == v) & (cvbr == cv))[0]
        o, l, _ = O.encode_streams(np.ascontiguousarray(pcm[idx]), FRAME, int(br), threads, vbr=int(v), cvbr=int(cv), complexity=10,
                                   max_bytes=stride, stride=stride, pin=False)
        out[idx] = o
        lens[idx] = l
    assert (lens > 2).all()
    return out, lens


def celt_header_flags(packets, lens):
    """(pf_on, transient) of CELT packets [m, stride] by decoding the first range-coded symbols (celt_decoder.c:850-887):
    silence (logp 15), post-filter flag (logp 1) [+ octave uniform(6), raw bits, tapset icdf], transient (logp 3)."""
    pf = np.zeros(len(lens), dtype=bool)
    tr = np.zeros(len(lens), dtype=bool)
    for k in range(len(lens)):
        d = packets[k, 1:lens[k]]           # skip the TOC
        pos = 0

        def byte():
            nonlocal pos
            b = int(d[pos]) if pos < len(d) else 0
            pos += 1
            return b
        rem = byte()
        rng = 128
        val = 127 - (rem >> 1)
        def norm():
            nonlocal rng, val, rem
            while rng <= (1 << 23):
                sym = rem
                rem = byte()
                sym = ((sym << 8) | rem) >> 1
                val = ((val << 8) + (255 & ~sym)) & 0x7FFFFFFF
                rng <<= 8
        norm()

        def bit_logp(logp):
            nonlocal rng, val
            s = rng >> logp
            r = val < s
            if not r:
                val -= s
                rng -= s
            else:
                rng = s
            norm()
            return r
        if bit_logp(15):
            continue
        if bit_logp(1):
            pf[k] = True
            # octave: ec_dec_uint(6)
            ft = 6
            s = rng // ft
            sym = ft - min(val // s + 1, ft)
            val -= s * (ft - (sym + 1))
            rng = s if sym > 0 else rng - s * (ft - 1)
            norm()
            # period and gain are raw bits (read from the end); tapset: ec_dec_icdf({2, 1, 0}, 2)
            r = rng >> 2
            s = rng
            for icdf in (2, 1, 0):
                t = s
                s = r * icdf
                if not val < s:
                    break
            val -= s
            rng = t - s
            norm()
        tr[k] = bit_logp(3)
    return pf, tr


class ClockSampler:
    """nvidia-smi sampler running during the timed region (B200_PROFILING.md 'clocks' line)."""

    def __init__(self, gpu_index):
        self.proc = None
        self.rows = []
        self.idx = gpu_index

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
            "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + q, "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for k, nm in enumerate(names):
                if len(r) > 4 + k and r[4 + k].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------------------------------------
# workload descriptions
# ------------------------------------------------------------------------------------------------------------------------------
def decode_config(args, world):
    return {"workload": "batched CELT decode: %d independent 48 kHz stereo 64 kbps CBR 20 ms streams per GPU, %d s each "
                        "(BASELINE.json configs[1])" % (args.streams, args.seconds),
            "streams_per_gpu": args.streams, "seconds_per_stream": args.seconds, "frame_ms": 20, "bitrate": BITRATE,
            "signals": "generate_music seed 13371337+s (clicks on 1/4), 1/8 of the streams from the reference's 48Khz Stereo.raw; "
                       "%d s unique per stream, repeated" % args.unique,
            "parallelism": "streams sharded over %d GPU(s), host partitioning, no collective" % world,
            "l2": "inputs+outputs per step (%.1f GB) >> 126 MB L2, no flush needed" % (args.streams * args.seconds * 50 * 4000 / 1e9)}


def encode_config(args, world):
    return {"workload": "batched CELT encode: %d independent 48 kHz stereo 96 kbps VBR complexity-10 20 ms streams per GPU, %d s each "
                        "(BASELINE.json configs[2])" % (args.streams, args.enc_seconds),
            "streams_per_gpu": args.streams, "seconds_per_stream": args.enc_seconds, "frame_ms": 20, "bitrate": ENC_BITRATE, "complexity": 10,
            "vbr": 1, "signals": "as the decode workload, %d s unique per stream" % min(args.unique, args.enc_seconds),
            "parallelism": "streams sharded over %d GPU(s), host partitioning, no collective" % world,
            "l2": "PCM in per step (%.1f GB) >> 126 MB L2, no flush needed" % (args.streams * args.enc_seconds * FS * CH * 2 / 1e9)}


def mixed_config(args, world):
    return {"workload": "mixed-bitrate decode + encode: %d streams in total sharded over %d GPU(s), 48 kHz stereo 20 ms, per-stream bitrate "
                        "drawn (seed 4) from %s bps, half CBR / half VBR, %d s each (BASELINE.json configs[4])"
                        % (args.mixed_streams, world, SWEEP_RATES, args.mixed_seconds),
            "streams_total": args.mixed_streams, "seconds_per_stream": args.mixed_seconds, "unique_programmes": args.mixed_unique,
            "scaling": "strong", "parallelism": "contiguous blocks of streams per GPU (concentus_b200/shard.py), no collective"}


def shard_range(n, rank, world):
    from concentus_b200.shard import shard_range as sr
    return sr(n, world, rank)


# ------------------------------------------------------------------------------------------------------------------------------
# the reference arm
# ------------------------------------------------------------------------------------------------------------------------------
def ref_lib(name="libopus_ref.so"):
    """oracle/_ref/<name>: the unmodified opus-fix build with oracle/ref_harness.c's thread pool; None when it was not built."""
    p = os.path.join(ROOT, "oracle", "_ref", name)
    if not os.path.exists(p):
        return None
    lib = C.CDLL(p)
    lib.ref_decode_streams_mt.restype = C.c_double
    lib.ref_decode_streams_mt.argtypes = [C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.ref_encode_streams_mt.restype = C.c_double
    lib.ref_encode_streams_mt.argtypes = [C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                          C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    return lib


def decode_input(n, seconds, unique, threads):
    """Packets of the first n streams of the decode workload: (blob, offs, lens, F)."""
    pcm = stream_signals(0, n, unique, threads)
    pk, lens = oracle_encode(pcm, BITRATE, 0, 0, threads, 256)
    plen = int(lens[0, 0])
    Fu = lens.shape[1]
    F = seconds * FS // FRAME
    reps = (F + Fu - 1) // Fu
    blob = np.ascontiguousarray(np.tile(pk[:, :, :plen], (1, reps, 1))[:, :F]).reshape(-1)
    return blob, np.arange(n * F, dtype=np.int64) * plen, np.full(n * F, plen, dtype=np.int32), F


def reference_decode(n, seconds, unique, threads, lib=None, inp=None):
    """The unmodified opus-fix decoder on the first n streams of the decode workload, one stream per thread.  (x realtime, wall s)"""
    import oracle_lib as O
    lib = lib or ref_lib()
    blob, offs, l2, F = inp if inp is not None else decode_input(n, seconds, unique, threads)
    t = lib.ref_decode_streams_mt(n, F, threads, O.ptr(blob), O.ptr(offs), O.ptr(l2), FRAME, CH, FS, None, None, None)
    return n * seconds / t, t


def reference_encode(n, seconds, unique, threads, lib=None):
    import oracle_lib as O
    lib = lib or ref_lib()
    u = min(unique, seconds)
    pcm = stream_signals(0, n, u, threads)
    reps = (seconds + u - 1) // u
    pcm = np.ascontiguousarray(np.tile(pcm, (1, reps, 1))[:, :seconds * FS])
    F = seconds * FS // FRAME
    out = np.zeros((n, F, 1276), dtype=np.uint8)
    lens = np.zeros((n, F), dtype=np.int32)
    cfg = O.RefEncCfg(O.OPUS_APPLICATION_RESTRICTED_LOWDELAY, ENC_BITRATE, 1, 0, 10, 1276, 0, 0)
    t = lib.ref_encode_streams_mt(n, F, threads, O.ptr(pcm), FRAME, CH, FS, C.byref(cfg), O.ptr(out), 1276, O.ptr(lens), None)
    assert (lens > 2).all()
    return n * seconds / t, t


def o3_lib():
    """oracle/_ref/libopus_ref_o3.so: the same unmodified sources at -O3 -march=x86-64-v3 (BASELINE.md section 3: 'so the comparison
    is not against a handicapped baseline'); None when it was not built."""
    return ref_lib("libopus_ref_o3.so")


def cpu_baselines(kind, n, seconds, unique, cores):
    """The reference on the host cores: -O2 as shipped, and -O3 -march=x86-64-v3 when built; None without the reference build."""
    if ref_lib() is None:
        return None
    fn = reference_decode if kind == "decode" else reference_encode
    v, t = fn(n, seconds, unique, cores)
    out = {"value": v, "unit": "x realtime", "cores": cores, "kind": "reference",
           "sample": "first %d streams x %d s of the workload, opus-fix -O2 build (the author's flags), one stream per thread, %.1f s wall" % (n, seconds, t)}
    lib = o3_lib()
    if lib is not None:
        v3, t3 = fn(n, seconds, unique, cores, lib)
        out["o3"] = {"value": v3, "flags": "-O3 -march=x86-64-v3", "wall_s": t3}
    return out


def run_reference(args, rank, world):
    if rank != 0:
        return
    if ref_lib() is None:
        raise SystemExit("bench.py --impl reference: oracle/_ref/libopus_ref.so not built (make -C oracle REF=<opus-fix source tree>)")
    cores = os.cpu_count() or 1
    n = min(args.streams, max(cores * 4, 16))
    sec = min(args.seconds, 30)
    inp = decode_input(n, sec, min(args.unique, sec), cores)
    vals = []
    for _ in range(args.warmup + args.steps):
        vals.append(reference_decode(n, sec, min(args.unique, sec), cores, inp=inp))
    vals = vals[args.warmup:]
    t = sum(v[1] for v in vals)
    val = n * sec * len(vals) / t
    enc_ref = None
    if not args.no_encode:
        ne = min(args.streams, max(cores * 16, 64))
        ev, et = reference_encode(ne, min(args.enc_seconds, 6), args.unique, cores)
        enc_ref = {"metric": ENC_METRIC, "value": ev, "unit": "x realtime", "config": encode_config(args, world),
                   "cpu_baseline": {"value": ev, "unit": "x realtime", "cores": cores, "kind": "reference",
                                    "sample": "%d streams x %d s, opus-fix -O2, one stream per thread, %.1f s wall" % (ne, min(args.enc_seconds, 6), et)}}
    line = {"impl": "reference", "encode": enc_ref, "metric": METRIC, "value": val, "unit": "x realtime", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * t / len(vals), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "int32", "data": "synthetic", "config": decode_config(args, world),
            "cpu_baseline": {"value": val, "unit": "x realtime", "cores": cores, "kind": "reference",
                             "sample": "%d streams x %d s (of %d streams x %d s per GPU), opus-fix -O2, one stream per thread" % (n, sec, args.streams, args.seconds)},
            "e2e": {"value": val, "unit": "x realtime", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------------------------------------
class Env:
    pass


def all_max(E, ms):
    if E.dist is None:
        return ms
    t = E.torch.tensor([ms], device=E.dev)
    E.dist.all_reduce(t, op=E.dist.ReduceOp.MAX)
    return float(t.item())


def barrier(E):
    E.torch.cuda.synchronize()
    E.L.opus_b200_synchronize()
    E.L.opus_b200_enc_synchronize()
    if E.dist is not None:
        E.dist.barrier()


DUMP_STREAMS, DUMP_FRAMES, DUMP_CAP = 32, 50, 64 << 20


def dump_window(S, F):
    """The fixed sample --dump-outputs writes: DUMP_STREAMS of the S streams and a window of DUMP_FRAMES of the F frames, seeded,
    so that its size does not grow with the workload (at most 12.3 MB of PCM or 8.2 MB of packets per workload)."""
    pick = np.sort(np.random.RandomState(1234).choice(S, min(DUMP_STREAMS, S), replace=False))
    nf = min(DUMP_FRAMES, F)
    f0 = int(np.random.RandomState(1235).randint(0, F - nf + 1))
    return pick, f0, nf


def dump_pcm(E, name, d_pcm, d_ret, S, F):
    """PCM [k, nf, FRAME*CH] and return codes [k, nf] of the sampled streams over the sampled frames."""
    pick, f0, nf = dump_window(S, F)
    sel = E.torch.from_numpy(pick).to(E.dev)
    E.dump[name + "_pcm"] = d_pcm.view(S, F, FRAME * CH)[sel, f0:f0 + nf].cpu().numpy().astype(np.float32)
    E.dump[name + "_ret"] = d_ret.view(S, F)[sel, f0:f0 + nf].cpu().numpy().astype(np.float32)
    E.dump[name + "_window"] = np.concatenate([pick, [f0, nf]]).astype(np.float64)   # stream indices, first frame, frame count


def dump_packets(E, name, d_data, d_ret, S, F, stride):
    """Packet bytes of the sampled streams over the sampled frames (concatenated in stream / frame order) and their lengths [k, nf]."""
    pick, f0, nf = dump_window(S, F)
    sel = E.torch.from_numpy(pick).to(E.dev)
    rows = d_data.view(S, F, stride)[sel, f0:f0 + nf].cpu().numpy()
    lens = d_ret.view(S, F)[sel, f0:f0 + nf].cpu().numpy()
    E.dump[name + "_packets"] = np.concatenate([rows[k, f, :max(int(lens[k, f]), 0)] for k in range(len(pick)) for f in range(nf)]).astype(np.float32)
    E.dump[name + "_lens"] = lens.astype(np.float32)
    E.dump[name + "_window"] = np.concatenate([pick, [f0, nf]]).astype(np.float64)


def input_digest(pk, lens):
    """Digest of a decode workload's packets (the oracle's encoding of its signals), so that runs can confirm identical inputs."""
    h = hashlib.blake2b(digest_size=8)
    for s in range(pk.shape[0]):
        for f in range(pk.shape[1]):
            h.update(pk[s, f, :max(int(lens[s, f]), 0)].tobytes())
    h.update(np.ascontiguousarray(lens, dtype=np.int32).tobytes())
    return h.hexdigest()


def F_chunk(F):
    for c in (1000, 750, 500, 250, 200, 100, 50, 25, 10, 5, 1):   # packets per e2e call: several pipeline chunks per call
        if F % c == 0:
            return c
    return 1


def bench_decode(E, args):
    import oracle_lib as O
    torch, L, cb, dev = E.torch, E.L, E.cb, E.dev
    S, seconds = args.streams, args.seconds
    F = seconds * FS // FRAME
    first = E.rank * S                                   # distinct streams on every GPU
    pcm = stream_signals(first, S, args.unique, E.threads)
    pk, lens_u = oracle_encode(pcm, BITRATE, 0, 0, E.threads, 256)
    del pcm
    digest = input_digest(pk, lens_u)
    plen = int(lens_u[0, 0])
    assert (lens_u == plen).all(), "CBR packets expected"
    Fu = lens_u.shape[1]
    fc = F_chunk(F)
    nchunks = F // fc
    # blob laid out [chunk][stream][frame-in-chunk] (one e2e call = one contiguous slab); frame f of a stream = its unique packet f % Fu
    fidx = np.arange(F) % Fu
    d_u = torch.from_numpy(np.ascontiguousarray(pk[:, :, :plen])).to(dev)                    # [S, Fu, plen]
    d_blob = d_u[:, torch.from_numpy(fidx).to(dev)].view(S, nchunks, fc, plen).permute(1, 0, 2, 3).contiguous().view(-1)
    del d_u
    c_idx = np.arange(F) // fc
    f_in = np.arange(F) % fc
    offs = ((c_idx[None, :] * S + np.arange(S)[:, None]) * fc + f_in[None, :]).astype(np.int64) * plen
    lens = np.full((S, F), plen, dtype=np.int32)
    d_offs = torch.from_numpy(offs.reshape(-1)).to(dev)
    d_lens = torch.from_numpy(lens.reshape(-1)).to(dev)
    d_pcm = torch.empty((S * F * FRAME * CH,), dtype=torch.int16, device=dev)
    d_ret = torch.zeros((S * F,), dtype=torch.int32, device=dev)
    dec = cb.DecoderBatch(S, FS, CH)
    stream = torch.cuda.ExternalStream(L.opus_b200_stream(), device=dev)

    def step_value(handles):
        rc = L.opus_decode_span_device(handles, S, F, C.c_void_p(d_blob.data_ptr()), C.c_void_p(d_offs.data_ptr()),
                                       C.c_void_p(d_lens.data_ptr()), C.c_void_p(d_pcm.data_ptr()), FRAME, C.c_void_p(d_ret.data_ptr()))
        assert rc == 0, rc

    for _ in range(args.warmup):
        step_value(dec.handles)
    barrier(E)
    L.opus_b200_stage_times(None, None, 1)
    sampler = ClockSampler(E.local)
    sampler.start()
    launches0 = L.opus_b200_kernel_launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        step_value(dec.handles)
    e1.record(stream)
    barrier(E)
    ms = all_max(E, e0.elapsed_time(e1))
    clocks = sampler.stop()
    assert bool((d_ret == FRAME).all().item()), "decode returned errors"
    if args.dump_outputs:
        dump_pcm(E, "decode", d_pcm, d_ret, S, F)
    launches = int(L.opus_b200_kernel_launches() - launches0)
    stage_ms = (C.c_double * 3)()
    stage_n = (C.c_longlong * 3)()
    L.opus_b200_stage_times(stage_ms, stage_n, 0)
    value = E.world * S * seconds * args.steps / (ms / 1e3)
    # roofline of the dominant kernel: algorithmic bytes = packet + PCM bytes of the frames one launch covers (SURVEY.md 8d:
    # 160 + 3,840 = 4,000 B per 20 ms stereo frame @ 64 kbps) over the kernel's mean launch duration (CUDA events on its stream)
    algo_step = float(lens.sum()) + float(S) * F * FRAME * CH * 2
    names = ["parse_kernel", "synth_kernel", "deemph_kernel"]
    stages = {}
    for i, nm in enumerate(names):
        n_l = int(stage_n[i])
        stages[nm] = {"launches": n_l, "ms_total": float(stage_ms[i]), "ms_per_launch": float(stage_ms[i]) / max(n_l, 1),
                      "share_of_stage_time": float(stage_ms[i]) / max(sum(stage_ms), 1e-9)}
    dom = max(names, key=lambda k: stages[k]["ms_total"])
    algo_launch = algo_step * args.steps / max(stages[dom]["launches"], 1)
    peak = float(E.peaks.get("hbm_gbs", 6650.0))
    achieved = algo_launch / (stages[dom]["ms_per_launch"] / 1e3) / 1e9
    traffic = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "decode_traffic.json")))
        traffic = tj["dram_bytes_per_frame"][dom] * (algo_launch / 4000.0)
    except Exception:
        pass
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "kernel": dom, "kernel_ms_per_launch": stages[dom]["ms_per_launch"], "algorithmic_bytes_per_launch": algo_launch, "stages": stages,
                "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if E.peaks else "fallback 6650 GB/s (of fallback)",
                "note": "integer-issue / latency bound path (SURVEY.md 8d).  `achieved` divides the PIPELINE's compulsory bytes (packets in + PCM out) by "
                        "the dominant kernel's time alone — stage A writes no PCM itself — as the contract's per-unit figure asks; limiter evidence "
                        "(issue utilisation, divergence, stall reasons) is under profiles/"}

    # ---- parity at the bench's full size (untimed): fresh decoders, the same device-resident call, 64 streams against the oracle ----
    parity = None
    if E.rank == 0 and not args.no_parity:
        decp = cb.DecoderBatch(S, FS, CH)
        step_value(decp.handles)
        barrier_local(E)
        pick = sorted(set(np.linspace(0, S - 1, args.parity_streams).astype(int).tolist()))
        rows = d_pcm.view(S, F * FRAME * CH)[torch.tensor(pick, device=dev)].cpu().numpy()
        fr = decp.final_ranges()
        nsel = len(pick)
        blob_sel = np.ascontiguousarray(np.tile(pk[pick][:, :, :plen], (1, (F + Fu - 1) // Fu, 1))[:, :F]).reshape(-1)
        o2 = np.arange(nsel * F, dtype=np.int64) * plen
        l2 = np.full(nsel * F, plen, dtype=np.int32)
        rp, rr, rret = O.decode_streams(nsel, F, E.threads, blob_sel, o2, l2, FRAME, CH, FS, pin=False)
        rp = rp.reshape(nsel, -1)
        bad = [int(s) for k, s in enumerate(pick)
               if not (np.array_equal(rp[k], rows[k]) and int(rr[(k + 1) * F - 1]) == int(fr[s]) and (rret[k * F:(k + 1) * F] == FRAME).all())]
        decp.close()
        parity = {"streams_checked": nsel, "packets_each": int(F), "mismatching_streams": bad,
                  "against": "the host simulation of the same codec headers (tests/oracle_lib.py, pin=False), fresh state, PCM sample-for-sample + final range"}
        assert not bad, "decode parity failed at bench size: streams %s" % bad

    # ---- e2e: host buffers through opus_decode_span (H2D + kernels + D2H per call) ----
    e2e = None
    if not args.no_e2e:
        del d_pcm
        torch.cuda.empty_cache()
        h_blob = d_blob.cpu().pin_memory()
        chunk_bytes = S * fc * plen
        h_pcm = torch.empty((S * fc * FRAME * CH,), dtype=torch.int16).pin_memory()
        h_ret = torch.empty((S * fc,), dtype=torch.int32).pin_memory()
        offs_c = np.ascontiguousarray((np.arange(S)[:, None] * fc + np.arange(fc)[None, :]).astype(np.int64) * plen).reshape(-1)
        lens_c = np.full(S * fc, plen, dtype=np.int32)
        dec2 = cb.DecoderBatch(S, FS, CH)

        def step_e2e():
            for c in range(nchunks):
                rc = L.opus_decode_span(dec2.handles, S, fc, C.c_void_p(h_blob.data_ptr() + c * chunk_bytes), cb._p(offs_c), cb._p(lens_c),
                                        C.c_void_p(h_pcm.data_ptr()), FRAME, C.c_void_p(h_ret.data_ptr()))
                assert rc == 0, rc
        for _ in range(args.warmup):
            step_e2e()
        barrier(E)
        t0 = time.perf_counter()
        e0.record(stream)
        for _ in range(args.steps):
            step_e2e()
        e1.record(stream)
        barrier(E)
        ems = all_max(E, max(e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3))
        assert bool((h_ret == FRAME).all().item())
        d2h = int(nchunks * (h_pcm.numel() * 2 + h_ret.numel() * 4))
        e2e = {"value": E.world * S * seconds * args.steps / (ems / 1e3), "unit": "x realtime",
               "h2d_bytes_per_step": int(h_blob.numel() + nchunks * (offs_c.nbytes + lens_c.nbytes)), "d2h_bytes_per_step": d2h,
               "ms_per_step": ems / args.steps, "d2h_gbs_per_gpu": d2h * args.steps / (ems / 1e3) / 1e9,
               "api": "opus_decode_span, %d calls of %d packets x %d streams per step, pinned host buffers" % (nchunks, fc, S)}
        dec2.close()
        del h_blob, h_pcm
    cpu = None
    if E.rank == 0 and E.world == 1 and not args.no_cpu:
        cpu = cpu_baselines("decode", min(S, max(E.cores * 8, 32)), min(seconds, 30), min(args.unique, seconds), E.cores)
    dec.close()
    del d_blob
    torch.cuda.empty_cache()
    return {"value": value, "ms": ms, "clocks": clocks, "launches": launches, "roofline": roofline, "parity": parity, "e2e": e2e, "cpu": cpu,
            "input_digest": digest}


def barrier_local(E):
    E.torch.cuda.synchronize()
    E.L.opus_b200_synchronize()
    E.L.opus_b200_enc_synchronize()


def bench_encode(E, args):
    """BASELINE.json configs[2] through opus_encode_span_device (value) and opus_encode_span (e2e)."""
    import oracle_lib as O
    torch, L, cb, dev = E.torch, E.L, E.cb, E.dev
    S, seconds = args.streams, args.enc_seconds
    F = seconds * FS // FRAME
    u = min(args.unique, seconds)
    first = E.rank * S
    pcm_u = stream_signals(first, S, u, E.threads)                            # [S, u*FS, CH]
    d_u = torch.from_numpy(pcm_u).to(dev)
    reps = (seconds + u - 1) // u
    d_pcm = d_u.repeat(1, reps, 1)[:, :seconds * FS].contiguous()
    del d_u
    stride = 1276
    d_data = torch.zeros((S * F * stride,), dtype=torch.uint8, device=dev)
    d_ret = torch.zeros((S * F,), dtype=torch.int32, device=dev)
    mk = lambda: cb.EncoderBatch(S, FS, CH, bitrate=ENC_BITRATE, vbr=1, cvbr=0, complexity=10)
    enc = mk()
    estream = torch.cuda.ExternalStream(L.opus_b200_enc_stream(), device=dev)

    def step_value(handles):
        rc = L.opus_encode_span_device(handles, S, F, C.c_void_p(d_pcm.data_ptr()), FRAME, C.c_void_p(d_data.data_ptr()), stride,
                                       C.c_void_p(d_ret.data_ptr()))
        assert rc == 0, rc

    for _ in range(args.warmup):
        step_value(enc.handles)
    barrier(E)
    launches0 = L.opus_b200_enc_kernel_launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(estream)
    for _ in range(args.steps):
        step_value(enc.handles)
    e1.record(estream)
    barrier(E)
    ms = all_max(E, e0.elapsed_time(e1))
    launches = int(L.opus_b200_enc_kernel_launches() - launches0)
    assert bool((d_ret > 2).all().item()), "encode returned errors"
    mean_len = float(d_ret.float().mean().item())
    if args.dump_outputs:
        dump_packets(E, "encode", d_data, d_ret, S, F, stride)
    value = E.world * S * seconds * args.steps / (ms / 1e3)
    pc, lc = C.c_longlong(0), C.c_longlong(0)
    L.opus_b200_enc_path_counts(C.byref(pc), C.byref(lc))
    # roofline: algorithmic bytes = PCM in + packet bytes out (SURVEY.md 8d: 3,840 + len per frame) over the span's device time; the
    # frame-synchronous pipeline has no single dominant kernel (profiles/r2_enc_launches_*.md), so the span is the unit
    algo = float(S) * F * (FRAME * CH * 2 + mean_len)
    peak = float(E.peaks.get("hbm_gbs", 6650.0))
    kms = ms / args.steps
    achieved = algo / (kms / 1e3) / 1e9
    traffic = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "encode_traffic.json")))
        traffic = tj["dram_bytes_per_frame"]["pipeline"] * S * F
    except Exception:
        pass
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "kernel": "encoder pipeline (one span = %d launches)" % (launches // max(args.steps, 1)), "kernel_ms_per_launch": kms,
                "algorithmic_bytes_per_launch": algo,
                "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if E.peaks else "fallback 6650 GB/s (of fallback)",
                "note": "integer-issue bound (every stage has all streams resident and issues at 45-70 % of the schedulers' slots); limiter "
                        "evidence per kernel under profiles/",
                "paths": {"pipeline_streams": int(pc.value), "one_kernel_streams": int(lc.value)}}
    # ---- parity at the bench's full size (untimed): fresh encoders, the same call, sampled streams against the oracle ----
    parity = None
    stats = None
    if E.rank == 0 and not args.no_parity:
        encp = mk()
        step_value(encp.handles)
        barrier_local(E)
        pick = sorted(set(np.linspace(0, S - 1, args.parity_streams).astype(int).tolist()))
        sel = torch.tensor(pick, device=dev)
        got_d = d_data.view(S, F, stride)[sel].cpu().numpy()
        got_l = d_ret.view(S, F)[sel].cpu().numpy()
        src = np.ascontiguousarray(d_pcm[sel].cpu().numpy())
        fr = encp.final_ranges()
        nsel = len(pick)
        rd, rl, rr = O.encode_streams(src, FRAME, ENC_BITRATE, E.threads, vbr=1, cvbr=0, complexity=10, max_bytes=1276, stride=1276, pin=False)
        bad = []
        for k, sidx in enumerate(pick):
            ok = np.array_equal(rl[k], got_l[k]) and all(np.array_equal(rd[k, f, :rl[k, f]], got_d[k, f, :rl[k, f]]) for f in range(F)) \
                and int(rr[k, -1]) == int(fr[sidx])
            if not ok:
                bad.append(int(sidx))
        encp.close()
        parity = {"streams_checked": nsel, "frames_each": int(F), "mismatching_streams": bad,
                  "against": "the host simulation of the same codec headers (tests/oracle_lib.py, pin=False), fresh state, packets byte-for-byte + final range"}
        assert not bad, "encode parity failed at bench size: streams %s" % bad
        # SURVEY.md 8d.3: the workload must exercise the pre-filter and the transient / short-MDCT paths: shares of the oracle's frames
        pf, tr = celt_header_flags(rd.reshape(-1, 1276), rl.reshape(-1))
        stats = {"frames": int(len(pf)), "pf_on_share": float(pf.mean()), "transient_share": float(tr.mean()),
                 "note": "post-filter flag / transient flag of the oracle's packets for the %d parity streams" % nsel}

    # ---- e2e: pinned host PCM in, host packets out, one opus_encode_span call per second of audio ----
    e2e = None
    if not args.no_e2e:
        del d_data
        torch.cuda.empty_cache()
        fc = FS // FRAME
        h_pcm = torch.empty((S, fc * FRAME, CH), dtype=torch.int16).pin_memory()
        h_pcm.copy_(d_pcm[:, :fc * FRAME].cpu())
        h_data = torch.empty((S * fc * stride,), dtype=torch.uint8).pin_memory()
        h_ret = torch.empty((S * fc,), dtype=torch.int32).pin_memory()
        enc2 = mk()

        def step_e2e():
            for c in range(seconds):
                rc = L.opus_encode_span(enc2.handles, S, fc, C.c_void_p(h_pcm.data_ptr()), FRAME, C.c_void_p(h_data.data_ptr()), stride,
                                        C.c_void_p(h_ret.data_ptr()))
                assert rc == 0, rc
        for _ in range(max(1, args.warmup - 2)):
            step_e2e()
        barrier(E)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            step_e2e()
        barrier(E)
        ems = all_max(E, (time.perf_counter() - t0) * 1e3)
        assert bool((h_ret > 2).all().item())
        e2e = {"value": E.world * S * seconds * args.steps / (ems / 1e3), "unit": "x realtime",
               "h2d_bytes_per_step": int(seconds * h_pcm.numel() * 2), "d2h_bytes_per_step": int(seconds * (h_data.numel() + h_ret.numel() * 4)),
               "ms_per_step": ems / args.steps,
               "api": "opus_encode_span, %d calls of %d frames x %d streams per step, pinned host buffers, wall clock" % (seconds, fc, S)}
        enc2.close()
    cpu = None
    if E.rank == 0 and E.world == 1 and not args.no_cpu:
        cpu = cpu_baselines("encode", min(S, max(E.cores * 16, 64)), min(seconds, 6), args.unique, E.cores)
    enc.close()
    del d_pcm
    torch.cuda.empty_cache()
    return {"metric": ENC_METRIC, "value": value, "unit": "x realtime", "ms_per_step": ms / args.steps,
            "mean_packet_bytes": mean_len, "config": encode_config(args, E.world), "e2e": e2e, "gpu_launches": launches,
            "roofline": roofline, "cpu_baseline": cpu, "parity": parity, "workload_stats": stats}


def bench_mixed(E, args):
    """BASELINE.json configs[4]: 65,536 streams in total with per-stream bitrate / CBR-VBR, decode and encode, sharded over the GPUs
    (strong scaling).  Inputs: `--mixed-unique` programmes (distinct seed and settings), replicated over the streams with a per-stream
    frame rotation; packets for the decode half come from the oracle."""
    import oracle_lib as O
    torch, L, cb, dev = E.torch, E.L, E.cb, E.dev
    NT, seconds, U = args.mixed_streams, args.mixed_seconds, min(args.mixed_unique, args.mixed_streams)
    lo, hi = shard_range(NT, E.rank, E.world)
    S = hi - lo
    F = seconds * FS // FRAME
    rs = np.random.RandomState(4)
    br_u = np.array(SWEEP_RATES)[rs.randint(len(SWEEP_RATES), size=U)]
    vbr_u = rs.randint(2, size=U)
    pcm_u = stream_signals(100000, U, seconds, E.threads)                     # [U, T, CH]
    pk_u, len_u = oracle_encode(pcm_u, br_u, vbr_u, 0, E.threads, 1276)       # [U, F, 1276]
    digest = input_digest(pk_u, len_u)
    prog = (np.arange(lo, hi) % U)
    rot = ((np.arange(lo, hi) // U) * 7) % F
    fidx = (np.arange(F)[None, :] + rot[:, None]) % F                         # [S, F]
    # ---- decode half: packed blob of the streams' (rotated) packet sequences ----
    lens = len_u[prog[:, None], fidx].astype(np.int32)                        # [S, F]
    offs = np.zeros(S * F, dtype=np.int64)
    offs[1:] = np.cumsum(lens.reshape(-1)[:-1])
    total = int(lens.sum())
    d_pk = torch.from_numpy(pk_u).to(dev)
    d_len_u = torch.from_numpy(len_u).to(dev)
    d_prog = torch.from_numpy(prog).to(dev)
    d_fidx = torch.from_numpy(fidx).to(dev)
    d_blob = torch.empty((total + 16,), dtype=torch.uint8, device=dev)
    d_offs = torch.from_numpy(offs).to(dev)
    d_lens = torch.from_numpy(lens.reshape(-1)).to(dev)
    col = torch.arange(1276, device=dev)
    for s0 in range(0, S, 256):                                                # pack on the device in slabs
        s1 = min(S, s0 + 256)
        rows = d_pk[d_prog[s0:s1, None], d_fidx[s0:s1]]                       # [s, F, 1276]
        ll = d_len_u[d_prog[s0:s1, None], d_fidx[s0:s1]]                      # [s, F]
        mask = col[None, None, :] < ll[:, :, None]
        d_blob[int(offs[s0 * F]):int(offs[s0 * F]) + int(ll.sum().item())] = rows[mask]
    del d_pk
    d_pcm = torch.empty((S * F * FRAME * CH,), dtype=torch.int16, device=dev)
    d_ret = torch.zeros((S * F,), dtype=torch.int32, device=dev)
    dec = cb.DecoderBatch(S, FS, CH)
    stream = torch.cuda.ExternalStream(L.opus_b200_stream(), device=dev)

    def dec_step():
        rc = L.opus_decode_span_device(dec.handles, S, F, C.c_void_p(d_blob.data_ptr()), C.c_void_p(d_offs.data_ptr()), C.c_void_p(d_lens.data_ptr()),
                                       C.c_void_p(d_pcm.data_ptr()), FRAME, C.c_void_p(d_ret.data_ptr()))
        assert rc == 0, rc
    dec_step()
    barrier(E)
    assert bool((d_ret == FRAME).all().item())
    # parity (the first launch decoded from fresh states): the first copy of a few programmes (rotation 0) against the oracle
    parity = None
    if E.rank == 0 and not args.no_parity:
        pick = [s for s in np.linspace(0, min(S, U) - 1, min(16, S)).astype(int).tolist() if rot[s] == 0]
        rows = d_pcm.view(S, F * FRAME * CH)[torch.tensor(pick, device=dev)].cpu().numpy()
        bad = []
        for k, s in enumerate(pick):
            u_ = int(prog[s])
            blob_s = np.ascontiguousarray(pk_u[u_]).reshape(-1)
            rp, _, rret = O.decode_stream(blob_s, np.arange(F, dtype=np.int64) * 1276, len_u[u_], FRAME, CH, pin=False)
            if not (np.array_equal(rp.reshape(-1), rows[k]) and (rret == FRAME).all()):
                bad.append(int(lo + s))
        parity = {"decode_streams_checked": len(pick), "decode_mismatching": bad}
        assert not bad, "mixed decode parity failed: %s" % bad
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        dec_step()
    e1.record(stream)
    barrier(E)
    dms = all_max(E, e0.elapsed_time(e1))
    if args.dump_outputs:
        dump_pcm(E, "mixed_decode", d_pcm, d_ret, S, F)
    dec_value = NT * seconds * args.steps / (dms / 1e3)
    dec.close()
    del d_blob, d_pcm
    torch.cuda.empty_cache()
    # ---- encode half: every stream with its own bitrate / VBR setting ----
    d_pu = torch.from_numpy(pcm_u).to(dev)                                     # [U, T, CH]
    d_in = torch.empty((S, F * FRAME, CH), dtype=torch.int16, device=dev)
    for s0 in range(0, S, 256):
        s1 = min(S, s0 + 256)
        t_idx = (torch.arange(F * FRAME, device=dev)[None, :] + (d_fidx[s0:s1, 0] * FRAME)[:, None]) % (F * FRAME)
        d_in[s0:s1] = d_pu[d_prog[s0:s1, None], t_idx]
    del d_pu
    stride = 1276
    d_data = torch.zeros((S * F * stride,), dtype=torch.uint8, device=dev)
    enc = cb.EncoderBatch(S, FS, CH, bitrate=ENC_BITRATE, vbr=1, cvbr=0, complexity=10)
    for i in range(S):
        hp = C.c_void_p(enc.handles[i])
        L.opus_encoder_ctl(hp, cb.OPUS_SET_BITRATE_REQUEST, C.c_int32(int(br_u[prog[i]])))
        L.opus_encoder_ctl(hp, cb.OPUS_SET_VBR_REQUEST, C.c_int32(int(vbr_u[prog[i]])))
    estream = torch.cuda.ExternalStream(L.opus_b200_enc_stream(), device=dev)

    def enc_step():
        rc = L.opus_encode_span_device(enc.handles, S, F, C.c_void_p(d_in.data_ptr()), FRAME, C.c_void_p(d_data.data_ptr()), stride,
                                       C.c_void_p(d_ret.data_ptr()))
        assert rc == 0, rc
    enc_step()
    barrier(E)
    assert bool((d_ret > 2).all().item())
    if E.rank == 0 and not args.no_parity:
        # the first launch coded fresh states: streams with rotation 0 must reproduce the oracle's packets of their programme
        pick = [s for s in np.linspace(0, min(S, U) - 1, min(16, S)).astype(int).tolist() if rot[s] == 0]
        sel = torch.tensor(pick, device=dev)
        got_d = d_data.view(S, F, stride)[sel].cpu().numpy()
        got_l = d_ret.view(S, F)[sel].cpu().numpy()
        bad = []
        for k, s in enumerate(pick):
            u_ = int(prog[s])
            if not (np.array_equal(len_u[u_], got_l[k]) and all(np.array_equal(pk_u[u_, f, :len_u[u_, f]], got_d[k, f, :len_u[u_, f]]) for f in range(F))):
                bad.append(int(lo + s))
        parity["encode_streams_checked"] = len(pick)
        parity["encode_mismatching"] = bad
        parity["against"] = "the host simulation of the same codec headers (tests/oracle_lib.py, pin=False): PCM sample-for-sample / packets byte-for-byte, fresh state"
        assert not bad, "mixed encode parity failed: %s" % bad
    e0.record(estream)
    for _ in range(args.steps):
        enc_step()
    e1.record(estream)
    barrier(E)
    ems = all_max(E, e0.elapsed_time(e1))
    if args.dump_outputs:
        dump_packets(E, "mixed_encode", d_data, d_ret, S, F, stride)
    enc_value = NT * seconds * args.steps / (ems / 1e3)
    enc.close()
    del d_in, d_data
    torch.cuda.empty_cache()
    cpu = None
    if E.rank == 0 and E.world == 1 and not args.no_cpu and ref_lib() is not None:
        nd = min(U, max(E.cores * 8, 32))
        blob = np.ascontiguousarray(pk_u[:nd]).reshape(-1)
        o2 = np.arange(nd * F, dtype=np.int64) * 1276
        l2 = np.ascontiguousarray(len_u[:nd]).reshape(-1)
        td = ref_lib().ref_decode_streams_mt(nd, F, E.cores, O.ptr(blob), O.ptr(o2), O.ptr(l2), FRAME, CH, FS, None, None, None)
        te = 0.0
        for (br, v) in sorted(set(zip(br_u[:nd].tolist(), vbr_u[:nd].tolist()))):   # one setting per call
            idx = np.nonzero((br_u[:nd] == br) & (vbr_u[:nd] == v))[0]
            cfg = O.RefEncCfg(O.OPUS_APPLICATION_RESTRICTED_LOWDELAY, int(br), int(v), 0, 10, 1276, 0, 0)
            o = np.zeros((len(idx), F, 1276), dtype=np.uint8)
            l = np.zeros((len(idx), F), dtype=np.int32)
            te += ref_lib().ref_encode_streams_mt(len(idx), F, E.cores, O.ptr(np.ascontiguousarray(pcm_u[idx])), FRAME, CH, FS, C.byref(cfg),
                                                  O.ptr(o), 1276, O.ptr(l), None)
        cpu = {"decode": nd * seconds / td, "encode": nd * seconds / te, "unit": "x realtime", "cores": E.cores, "kind": "reference",
               "sample": "%d of the %d programmes x %d s, opus-fix -O2, one stream per thread" % (nd, U, seconds)}
    return {"metric": "CELT mixed-bitrate decode / encode audio-sec per sec (x realtime), 48k stereo, %d streams" % NT,
            "decode": {"value": dec_value, "unit": "x realtime", "ms_per_step": dms / args.steps},
            "encode": {"value": enc_value, "unit": "x realtime", "ms_per_step": ems / args.steps},
            "streams_this_rank": int(S), "scaling": "strong", "input_digest": digest, "config": mixed_config(args, E.world), "parity": parity, "cpu_baseline": cpu}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--streams", type=int, default=4096, help="streams per GPU")
    ap.add_argument("--seconds", type=int, default=60, help="audio seconds per stream per decode step")
    ap.add_argument("--unique", type=int, default=6, help="seconds of distinct signal per stream (repeated to the workload's length)")
    ap.add_argument("--enc-seconds", type=int, default=6, help="audio seconds per stream per encode step")
    ap.add_argument("--mixed-streams", type=int, default=65536, help="streams in total of the mixed-bitrate workload (configs[4])")
    ap.add_argument("--mixed-seconds", type=int, default=2)
    ap.add_argument("--mixed-unique", type=int, default=1024, help="distinct (signal, settings) programmes of the mixed workload")
    ap.add_argument("--parity-streams", type=int, default=64)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-encode", action="store_true")
    ap.add_argument("--no-mixed", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the untimed full-size parity passes against the oracle")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the timed calls returned in their last step to DIR/<name>.npy")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import concentus_b200 as cb
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the CELT engine has no CPU path")
    torch.cuda.set_device(local)
    E = Env()
    E.torch, E.cb, E.rank, E.world, E.local = torch, cb, rank, world, local
    E.dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        E.dist = dist
    E.L = cb.lib()
    assert E.L.opus_b200_init(local) == 0
    E.dev = torch.device("cuda", local)
    E.cores = os.cpu_count() or 1
    E.threads = max(1, E.cores // max(world, 1))
    E.peaks = {}
    E.dump = {}
    try:
        E.peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass

    d = bench_decode(E, args)
    launches = d["launches"]
    encode = None
    if not args.no_encode:
        encode = bench_encode(E, args)
        launches += encode["gpu_launches"]
    mixed = None
    if not args.no_mixed:
        mixed = bench_mixed(E, args)
    if rank == 0:
        line = {"metric": METRIC, "value": d["value"], "unit": "x realtime", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": d["ms"] / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32",
                "data": "synthetic", "config": decode_config(args, world), "clocks": d["clocks"], "e2e": d["e2e"], "gpu_launches": int(launches),
                "roofline": d["roofline"], "cpu_baseline": d["cpu"], "parity": d["parity"], "input_digest": d["input_digest"],
                "encode": encode, "mixed": mixed}
        print(json.dumps(line), flush=True)
        if args.dump_outputs:
            assert sum(a.nbytes for a in E.dump.values()) <= DUMP_CAP, "--dump-outputs: sample larger than 64 MB"
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, a in E.dump.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    if E.dist is not None:
        E.dist.destroy_process_group()


if __name__ == "__main__":
    main()

"""The reference's OWN programs on the GPU path (VERDICT r1 item 3): opus-fix/src/opus_demo.c, tests/test_opus_padding.c,
tests/test_opus_decode.c and tests/test_opus_api.c, compiled from the reference's unmodified sources against the reference's
headers and linked to libconcentus_b200.so by the committed recipe oracle/Makefile (target `b200`; the decode test is restricted
to the CELT configurations and the API test loses its multistream sections through the committed sed scripts
oracle/celt_only_decode.sed / oracle/no_multistream_api.sed).  The reference's sources are not part of this repository: the
binaries exist only where `make -C oracle REF=<opus-fix source tree>` was run, and these tests skip elsewhere."""
import os
import subprocess

import numpy as np
import pytest

import oracle_lib as O

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, "oracle", "_ref")


def _need(name):
    p = os.path.join(REF, name)
    if not os.path.exists(p):
        pytest.skip("oracle/_ref/%s not built: needs the reference's sources (make -C oracle REF=<opus-fix source tree>)" % name)
    return p


def _run(args, timeout):
    return subprocess.run(args, cwd=REF, capture_output=True, text=True, timeout=timeout)


def test_opus_demo_on_our_library_matches_the_oracle_byte_for_byte(tmp_path):
    """BASELINE.json configs[0]: opus_demo restricted-lowdelay 48000 2 128000 -complexity 10 -framesize 20 on the 10 s generate_music
    signal.  The .bit file written by the reference's opus_demo linked to OUR library must be identical to the one written by the
    reference's opus_demo on its own library; the same for the decoded PCM (both directions through the scalar libopus API)."""
    ours, ref = _need("opus_demo_b200"), _need("opus_demo")
    pcm = O.generate_music(480000, 13371337)
    raw = tmp_path / "music10s.raw"
    pcm.astype("<i2").tofile(raw)
    enc_args = ["-e", "restricted-lowdelay", "48000", "2", "128000", "-complexity", "10", "-framesize", "20", str(raw)]
    r = _run([ref] + enc_args + [str(tmp_path / "ref.bit")], 300)
    assert r.returncode == 0, r.stderr[-400:]
    r = _run([ours] + enc_args + [str(tmp_path / "ours.bit")], 600)
    assert r.returncode == 0, (r.stdout[-400:], r.stderr[-400:])
    a, b = (tmp_path / "ref.bit").read_bytes(), (tmp_path / "ours.bit").read_bytes()
    assert len(a) > 100000 and a == b, "opus_demo -e on libconcentus_b200.so differs from the reference's .bit file"
    r = _run([ref, "-d", "48000", "2", str(tmp_path / "ref.bit"), str(tmp_path / "ref.pcm")], 300)
    assert r.returncode == 0, r.stderr[-400:]
    r = _run([ours, "-d", "48000", "2", str(tmp_path / "ref.bit"), str(tmp_path / "ours.pcm")], 600)
    assert r.returncode == 0, (r.stdout[-400:], r.stderr[-400:])
    a, b = (tmp_path / "ref.pcm").read_bytes(), (tmp_path / "ours.pcm").read_bytes()
    assert len(a) >= 480000 * 4 and a == b, "opus_demo -d on libconcentus_b200.so differs from the reference's PCM"
    # and the reference's default mode (encode + decode in one run, with its per-packet final-range check between the two)
    r = _run([ours, "restricted-lowdelay", "48000", "2", "96000", "-cvbr", "-framesize", "10", str(raw), str(tmp_path / "both.pcm")], 900)
    assert r.returncode == 0 and "Error: Range coder state mismatch" not in r.stderr, r.stderr[-400:]
    r2 = _run([ref, "restricted-lowdelay", "48000", "2", "96000", "-cvbr", "-framesize", "10", str(raw), str(tmp_path / "both_ref.pcm")], 300)
    assert r2.returncode == 0
    assert (tmp_path / "both.pcm").read_bytes() == (tmp_path / "both_ref.pcm").read_bytes()


def test_reference_padding_test_on_our_library():
    r = _run([_need("test_opus_padding_b200")], 300)
    assert r.returncode == 0 and "All padding tests passed" in r.stdout + r.stderr, (r.stdout[-300:], r.stderr[-300:])


def test_reference_api_test_on_our_library():
    """tests/test_opus_api.c minus multistream: every ctl / argument-validation / return code of the decoder, encoder, packet
    parser and repacketizer sections (6.7 M API invocations)."""
    r = _run([_need("test_opus_api_b200")], 900)
    out = r.stdout + r.stderr
    assert r.returncode == 0 and "All repacketizer tests passed" in out and "All encoder interface tests passed" in out \
        and "All decoder interface tests passed" in out, (r.stdout[-600:], r.stderr[-300:])


def test_reference_decode_test_on_our_library():
    """tests/test_opus_decode.c restricted to the CELT configurations: PLC on fresh decoders, all 2-byte prefixes, the cres[]
    known-answer sums of OPUS_GET_FINAL_RANGE over all 65,536 3-byte prefixes (tests/test_opus_decode.c:236-258), random packets of
    every size, all CELT mode pairs, the sentinel guard around the output buffer; 10 decoders (5 rates x 2
    channel counts) must agree on the final range.  The same filtered source passes on the reference library (checked at build)."""
    r = _run([_need("test_opus_decode_b200")], 1500)
    assert r.returncode == 0, (r.stdout[-600:], r.stderr[-300:])
    out = r.stdout + r.stderr
    assert "all 3-byte prefix for length 4, mode" in out and "all mode pairs (4096)*10" in out and "Decoders stopped" in out

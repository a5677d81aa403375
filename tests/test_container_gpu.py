"""GPU: batch file coding through the `.bit` container (concentus_b200/bitfile.py, SURVEY.md §8f rank 4), checked against what
the reference's own command-line codec (src/opus_demo.c) does with such files: it decodes the files our CUDA encoder wrote —
verifying the stored final range against its decoder on every packet (src/opus_demo.c:806-816) — and our CUDA decoder must
reproduce its output for files it wrote.  The reference's side is restated through the oracle (tests/oracle_lib.py)."""
import numpy as np
import pytest

import oracle_lib as O

pytestmark = pytest.mark.gpu


def _cb():
    import concentus_b200 as cb
    assert cb.lib().opus_b200_init(0) == 0, "CUDA device required: no CPU fallback exists"
    return cb


def _demo_decode(bit, ch, fs):
    """`opus_demo -d 48000 <ch> <bit> <out>`: every record decoded (length 0 = lost packet), the stored final range checked
    against the decoder's for every received packet, the samples of every packet written."""
    from concentus_b200 import bitfile
    data, offs, lens, ranges = bitfile.read_bit(str(bit))
    pcm, rng, rets = O.decode_stream(data, offs, lens, fs, ch)
    assert (rets == fs).all(), rets
    got = lens > 0
    assert np.array_equal(rng[got], ranges[got]), "Range coder state mismatch"
    return pcm


def _demo_encode(pcm, ch, fs, br, bit):
    """`opus_demo -e restricted-lowdelay 48000 <ch> <br> [-framesize <fs>] <raw> <bit>` (VBR, complexity 10): the input is coded
    in whole frames, zero-padded, with one extra frame when it ends on a frame boundary (src/opus_demo.c:672-690)."""
    from concentus_b200 import bitfile
    x = np.zeros(((len(pcm) // fs + 1) * fs, ch), dtype=np.int16)
    x[:len(pcm)] = pcm
    d, o, l, r = O.encode_stream(x, fs, br, ch, vbr=1, cvbr=0, complexity=10, max_bytes=1500)
    d, o = O.pack(d, o, l)
    bitfile.write_bit(str(bit), d, o, l, r)


@pytest.mark.parametrize("ch,fs,br", [(2, 960, 96000), (1, 480, 64000)])
def test_our_files_decode_in_the_reference_tool(tmp_path, ch, fs, br):
    _cb()
    from concentus_b200 import bitfile
    # ragged batch: three inputs of different length, one ending mid-frame
    pcms = [O.test_signal(48000, ch, 300, "music"), O.test_signal(24000 + 77, ch, 301, "tone"), O.test_signal(36000, ch, 302, "clicks")]
    paths = [str(tmp_path / ("s%d.bit" % i)) for i in range(3)]
    nf = bitfile.encode_files(pcms, paths, 48000, ch, fs, bitrate=br, vbr=1, cvbr=0, complexity=10)
    ours = bitfile.decode_files(paths, 48000, ch, fs)
    for i, p in enumerate(pcms):
        data, offs, lens, ranges = bitfile.read_bit(paths[i])
        assert len(lens) == nf[i] == len(p) // fs + 1
        # byte-for-byte what the reference encoder produces for opus_demo's zero-padded input
        x = np.zeros((nf[i] * fs, ch), dtype=np.int16)
        x[:len(p)] = p
        rd, ro, rl, rr = O.encode_stream(x, fs, br, ch, vbr=1, cvbr=0, complexity=10)
        assert np.array_equal(lens, rl) and np.array_equal(ranges, rr), i
        for f in range(nf[i]):
            assert np.array_equal(data[offs[f]:offs[f] + lens[f]], rd[ro[f]:ro[f] + rl[f]]), (i, f)
        # the reference tool accepts the file (range check on every packet) and decodes it to what our decoder gives
        ref = _demo_decode(paths[i], ch, fs)
        assert ref.shape == ours[i].shape and np.array_equal(ref, ours[i]), i


def test_reference_files_with_loss_decode_like_the_reference_tool(tmp_path):
    _cb()
    from concentus_b200 import bitfile
    ch, fs = 2, 960
    paths = []
    for i, (nsamp, br) in enumerate(((48000, 64000), (30000, 128000), (19200, 32000))):
        pcm = O.test_signal(nsamp, ch, 310 + i, ("music", "tone", "noise")[i])
        bit = tmp_path / ("r%d.bit" % i)
        _demo_encode(pcm, ch, fs, br, bit)
        if i == 1:   # knock packets out of the second file: length-0 records are lost packets (src/opus_demo.c:763)
            d, o, l, rg = bitfile.read_bit(str(bit))
            l = l.copy()
            l[5::9] = 0
            l[20:24] = 0
            bitfile.write_bit(str(bit), d, o, l, np.where(l > 0, rg, 0))
        paths.append(str(bit))
    ours = bitfile.decode_files(paths, 48000, ch, fs)
    for i, p in enumerate(paths):
        ref = _demo_decode(p, ch, fs)
        assert ref.shape == ours[i].shape and np.array_equal(ref, ours[i]), i

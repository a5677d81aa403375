"""The multistream encoder's side, in plain Python (no library code): how libopus's opus_multistream_encode frames each stream's
packet (the repacketizer), its rate allocation and its byte budgets (src/opus_multistream_encoder.c 1.1.x), on top of the packet
framing of ms_framing.py."""
from ms_framing import build, parse


def ms_frame(pkt, self_delimited, pad=False, maxlen=1 << 30):
    """What libopus's multistream encoder makes of one stream's ordinary packet (opus_repacketizer_cat + _out_range_impl): the
    frames re-framed with the cheapest frame-count code, the packet's own padding dropped, self-delimited for streams 0..S-2, and
    with `pad` padded to exactly maxlen.  Returns the bytes, or -2 (OPUS_BUFFER_TOO_SMALL) when they exceed maxlen."""
    toc, _, frames, _, _ = parse(pkt)
    cfg, lens = toc & 0xFC, [len(f) for f in frames]
    sd = (1 + (lens[-1] >= 252)) if self_delimited else 0
    if len(frames) == 1:
        code, header = 0, 1
    elif len(frames) == 2 and lens[0] == lens[1]:
        code, header = 1, 1
    elif len(frames) == 2:
        code, header = 2, 2 + (lens[0] >= 252)
    else:
        code, header = 3, 0
    if code != 3:
        total = header + sd + sum(lens)
        if total > maxlen:
            return -2
        if not (pad and total < maxlen):
            return build(cfg, code, frames, self_delimited=self_delimited)
    vbr = int(len(set(lens)) > 1)
    total = 2 + sd + (sum(1 + (n >= 252) for n in lens[:-1]) if vbr else 0) + sum(lens)
    if total > maxlen:
        return -2
    extra = maxlen - total if pad else 0
    return build(cfg, 3, frames, vbr=vbr, pad=extra, self_delimited=self_delimited)


def c_div(a, b):
    """C integer division (truncates towards zero)."""
    q = abs(a) // abs(b)
    return q if (a >= 0) == (b >= 0) else -q


def ms_rates(B, channels, streams, coupled, Fs, frame_size):
    """libopus's surround_rate_allocation without an LFE stream: each stream's bitrate for one call."""
    offset = 20000 if B > 40000 * channels else c_div(c_div(B, channels), 2)
    offset += 60 * (Fs // frame_size - 50)
    if B == -1000:
        ch = Fs + 60 * Fs // frame_size
    elif B == -1:
        ch = 300000
    else:
        ch = c_div(256 * (B - offset * streams), 256 * (streams - coupled) + 512 * coupled)
    return [offset + ((ch * 512) >> 8) if s < coupled else offset + ch for s in range(streams)]


def ms_budget(max_data_bytes, tot_size, streams, s):
    """The bytes stream s may take once the streams before it took tot_size (opus_multistream_encode_native)."""
    return min(max_data_bytes - tot_size - max(0, 4 * (streams - s - 1) - 1), 3 * 1275 + 7)


def ms_cbr_max_bytes(max_data_bytes, B, Fs, frame_size):
    return min(max_data_bytes, c_div(3 * B, 3 * 8 * Fs // frame_size))

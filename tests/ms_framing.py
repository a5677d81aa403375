"""Multistream packets for the tests, in plain Python (no library code): RFC 6716 §3.2 framing of ordinary Opus packets, the
self-delimiting variant of RFC 6716 Appendix B, and the multistream packet of RFC 7845 §5.1.1 / libopus opus_multistream.h
(streams 0..S-2 self-delimited, the last stream an ordinary packet)."""
import numpy as np


def size_bytes(n):
    """A frame length as a packet header writes it."""
    assert 0 <= n <= 1275
    if n < 252:
        return bytes([n])
    b0 = 252 + (n & 3)
    return bytes([b0, (n - b0) >> 2])


def parse(pkt):
    """An ordinary packet -> (toc, code, frames, vbr, padding bytes).  Valid packets only."""
    pkt = bytes(pkt)
    toc, code, p = pkt[0], pkt[0] & 3, 1

    def rd(p):
        if pkt[p] < 252:
            return pkt[p], p + 1
        return pkt[p] + 4 * pkt[p + 1], p + 2
    if code == 0:
        return toc, code, [pkt[1:]], 0, 0
    if code == 1:
        h = (len(pkt) - 1) // 2
        return toc, code, [pkt[1:1 + h], pkt[1 + h:]], 0, 0
    if code == 2:
        n0, p = rd(1)
        return toc, code, [pkt[p:p + n0], pkt[p + n0:]], 0, 0
    ch = pkt[1]
    count, vbr, padded = ch & 0x3F, (ch >> 7) & 1, (ch >> 6) & 1
    p, pad = 2, 0   # pad: padding data bytes
    if padded:
        while True:
            b = pkt[p]
            p += 1
            pad += 254 if b == 255 else b
            if b != 255:
                break
    pad_total = pad + (p - 2)   # as build() counts it: with the padding-length bytes
    body = len(pkt) - p - pad
    if vbr:
        sizes = []
        for _ in range(count - 1):
            n, p = rd(p)
            sizes.append(n)
        body = len(pkt) - p - pad
        sizes.append(body - sum(sizes))
    else:
        sizes = [body // count] * count
    frames, q = [], p
    for n in sizes:
        frames.append(pkt[q:q + n])
        q += n
    return toc, code, frames, vbr, pad_total


def build(toc_cfg, code, frames, vbr=None, pad=0, self_delimited=False):
    """Frames -> a packet with frame-count code `code` (code 3: CBR unless vbr, `pad` bytes of padding in all)."""
    frames = [bytes(f) for f in frames]
    out = bytearray([toc_cfg | code])
    if code == 0:
        assert len(frames) == 1
    elif code == 1:
        assert len(frames) == 2 and len(frames[0]) == len(frames[1])
    elif code == 2:
        assert len(frames) == 2
        out += size_bytes(len(frames[0]))
    else:
        if vbr is None:
            vbr = int(len({len(f) for f in frames}) > 1)
        out.append(len(frames) | (0x80 if vbr else 0) | (0x40 if pad else 0))
        if pad:
            # `pad` counts the padding-length bytes too (as libopus's opus_packet_pad does)
            n255 = (pad - 1) // 255
            out += bytes([255] * n255 + [pad - 255 * n255 - 1])
        if vbr:
            for f in frames[:-1]:
                out += size_bytes(len(f))
    if self_delimited:
        out += size_bytes(len(frames[-1]))
    for f in frames:
        out += f
    if code == 3 and pad:
        out += bytes(pad - ((pad - 1) // 255 + 1))
    return bytes(out)


def self_delimit(pkt):
    """An ordinary packet -> the same packet in self-delimiting framing (RFC 6716 Appendix B), padding kept."""
    toc, code, frames, vbr, pad = parse(pkt)
    return build(toc & 0xFC, code, frames, vbr=vbr, pad=pad, self_delimited=True)


def ms_packet(subpackets):
    """Ordinary packets of S streams -> one multistream packet."""
    return b"".join(self_delimit(p) for p in subpackets[:-1]) + bytes(subpackets[-1])


def pad_packet(pkt, extra):
    """Re-frame an ordinary packet as code 3 with `extra` bytes of padding (same frames)."""
    toc, code, frames, vbr, _ = parse(pkt)
    return build(toc & 0xFC, 3, frames, vbr=int(len({len(f) for f in frames}) > 1), pad=extra)


def ms_blob(packets):
    """A list of byte strings -> (uint8 blob, int64 offsets, int32 lengths)."""
    offs, lens, base = [], [], 0
    for p in packets:
        offs.append(base)
        lens.append(len(p))
        base += len(p)
    blob = np.frombuffer(b"".join(bytes(p) for p in packets) + b"\0", dtype=np.uint8).copy()
    return blob, np.array(offs, dtype=np.int64), np.array(lens, dtype=np.int32)

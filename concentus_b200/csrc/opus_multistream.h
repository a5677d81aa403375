// opus_multistream.h — the packet side of the multistream decoder and encoder, usable from host and device code.
//
// A multistream packet of S streams (RFC 7845 §5.1.1, libopus opus_multistream.h) carries one Opus packet per stream: streams
// 0..S-2 in self-delimited framing (RFC 6716 Appendix B), the last stream as an ordinary packet made of all remaining bytes.
// ms_split_packet validates such a packet the way opus_multistream_decode does before it decodes anything, and rewrites it as S
// ordinary packets that the single-stream decoder stages take unchanged.  ms_pack_packet is the encoder's inverse: it frames one
// stream's ordinary packet for its place in a multistream packet.
#pragma once
#include "opus_packet.h"

namespace cb {

// The elementary packet of every stream of a rejected multistream packet: a code-3 packet of zero frames.  pkt_parse rejects it
// (OPUS_INVALID_PACKET), so stage A marks the packet rejected and stage B leaves the state untouched; the multistream call reports
// the packet's own error code.  (A length <= 0 would not do: the stages read it as a lost packet and conceal.)
enum { kMsRejectLen = 2 };
CB_HD void ms_write_reject_marker(uint8_t *p) {
    p[0] = 0xFB;   // CELT fullband 20 ms, code 3
    p[1] = 0x00;   // zero frames
}

// Validates the multistream packet data[0..len) of S streams for a decoder at Fs with `frame_size` samples of room per channel:
//   len < 0: OPUS_BAD_ARG; len == 0: lost (every stream conceals); len < 2S-1: OPUS_INVALID_PACKET; then every sub-packet must
//   parse (else its parse error), all must carry the same number of samples (else OPUS_INVALID_PACKET) and that number must fit
//   in frame_size (else OPUS_BUFFER_TOO_SMALL).  A SILK or hybrid sub-packet that carries a frame is outside this decoder's scope:
//   OPUS_UNIMPLEMENTED, decided here so that no stream of the packet is decoded.
// On success the sub-packets of streams 0..S-2 are rewritten undelimited — TOC and frames with the same frame-count code, without
// the self-delimiting length or padding — into `out`, a copy of `data` (out[i] mirrors data[i]): the new header is never longer
// than the old one, so it ends where the sub-packet's frames begin and only the sub-packet's own header bytes are overwritten.
// The last stream's packet is used as it is.  Stream s's packet is then out[eoffs[s*estride] - base ..][0 .. elens[s*estride]).
// A lost packet gives elens = 0 in every stream.  A rejected one gives every stream the packet at `reject_off` (in the offsets'
// frame), which holds ms_write_reject_marker's bytes: the decoder stages reject it without touching state.
// Returns the samples per channel of the packet, 0 when it is lost, or the error code.
CB_HD int ms_split_packet(const uint8_t *data, int len, int S, int Fs, int frame_size, uint8_t *out, int64_t base, int64_t *eoffs,
                          int32_t *elens, size_t estride, int64_t reject_off) {
    int ret = 0;
    if (len < 0) {
        ret = -1;   // OPUS_BAD_ARG
    } else if (len > 0 && len < 2 * S - 1) {
        ret = -4;   // OPUS_INVALID_PACKET
    } else if (len > 0) {
        // opus_multistream_packet_validate: every sub-packet, before anything is decoded
        int16_t size[48];
        uint8_t toc;
        int rem = len, pos = 0, samples = 0, unimpl = 0;
        for (int s = 0; s < S && ret == 0; s++) {
            int poff = 0, pkoff = 0;
            if (rem <= 0) { ret = -4; break; }
            const int count = pkt_parse(data + pos, rem, s != S - 1, &toc, size, &poff, &pkoff);
            if (count < 0) { ret = count; break; }
            const int ns = count * pkt_samples_per_frame(data + pos, Fs);
            if (ns * 25 > Fs * 3 || (s > 0 && ns != samples)) { ret = -4; break; }
            samples = ns;
            if (pkt_mode(data + pos) != CB_MODE_CELT_ONLY)
                for (int i = 0; i < count; i++) unimpl |= size[i] > 1;
            pos += pkoff;
            rem -= pkoff;
        }
        if (ret == 0 && samples > frame_size) ret = -2;   // OPUS_BUFFER_TOO_SMALL
        if (ret == 0 && unimpl) ret = -5;                 // OPUS_UNIMPLEMENTED
        if (ret == 0) {
            rem = len;
            pos = 0;
            for (int s = 0; s < S; s++) {
                int poff = 0, pkoff = 0;
                const int count = pkt_parse(data + pos, rem, s != S - 1, &toc, size, &poff, &pkoff);
                if (s == S - 1) {
                    eoffs[s * estride] = base + pos;
                    elens[s * estride] = rem;
                    break;
                }
                const int code = toc & 3;
                const int vbr = code == 3 && (data[pos + 1] & 0x80);
                uint8_t hdr[2 + 47 * 2];
                const int hl = pkt_write_header(hdr, (uint8_t)(toc & 0xFC), code, count, vbr, 0, size);
                const int start = pos + poff - hl;
                for (int i = 0; i < hl; i++) out[start + i] = hdr[i];
                int bytes = hl;
                for (int i = 0; i < count; i++) bytes += size[i];
                eoffs[s * estride] = base + start;
                elens[s * estride] = bytes;
                pos += pkoff;
                rem -= pkoff;
            }
            return samples;
        }
    }
    for (int s = 0; s < S; s++) {
        eoffs[s * estride] = ret < 0 ? reject_off : base;
        elens[s * estride] = ret < 0 ? kMsRejectLen : 0;
    }
    return ret;
}

// The encoder's side: stream s's ordinary packet pkt[0..len) as it goes into a multistream packet, written to out[0..maxlen)
// (which must not overlap pkt).  This is opus_repacketizer_cat followed by opus_repacketizer_out_range_impl over all its frames
// (repacketizer.c:62-227): the frames are re-framed with the cheapest frame-count code (plan_layout), the packet's own padding
// is dropped, streams 0..S-2 are self-delimited (RFC 6716 Appendix B) and with `pad` (the last stream of a CBR call) the packet
// is padded to exactly maxlen.  Returns the bytes written or a negative error (the packet's parse error, OPUS_BUFFER_TOO_SMALL).
CB_HD int ms_pack_packet(const uint8_t *pkt, int len, int self_delimited, int pad, uint8_t *out, int maxlen) {
    int16_t size[48];
    uint8_t toc;
    int poff = 0;
    const int count = pkt_parse(pkt, len, 0, &toc, size, &poff, nullptr);
    if (count < 0) return count;
    const int sd = self_delimited ? 1 + (size[count - 1] >= 252) : 0;
    PktLayout L;
    const int rc = plan_layout(size, count, maxlen, pad, L, sd);
    if (rc < 0) return rc;
    uint8_t *q = out + pkt_write_header(out, (uint8_t)(toc & 0xFC), L.code, count, L.vbr, L.pad, size);
    if (self_delimited) q += pkt_put_size(size[count - 1], q);
    const uint8_t *src = pkt + poff;
    int payload = 0;
    for (int i = 0; i < count; i++) payload += size[i];
    for (int i = 0; i < payload; i++) *q++ = src[i];
    while (q < out + L.total) *q++ = 0;   // the padding bytes
    return L.total;
}

}  // namespace cb

// opus_packet.h — Opus packet framing (TOC byte, frame-count codes 0-3, padding), usable from host and
// device code.  Restates opus-fix/src/opus.c:148-343 (parse_size, opus_packet_get_samples_per_frame,
// opus_packet_parse_impl) and src/opus_decoder.c:185-198,921-975 (mode / bandwidth / channel getters).
#pragma once
#include <stdint.h>
#include "opus_state.h"

#if defined(__CUDACC__)
#define CB_HD __host__ __device__ inline
#else
#define CB_HD static inline
#endif

namespace cb {

CB_HD int pkt_mode(const uint8_t *d) {
    if (d[0] & 0x80) return CB_MODE_CELT_ONLY;
    if ((d[0] & 0x60) == 0x60) return CB_MODE_HYBRID;
    return CB_MODE_SILK_ONLY;
}
CB_HD int pkt_bandwidth(const uint8_t *d) {
    int bw;
    if (d[0] & 0x80) {
        bw = 1102 + ((d[0] >> 5) & 0x3);
        if (bw == 1102) bw = 1101;
    } else if ((d[0] & 0x60) == 0x60) {
        bw = (d[0] & 0x10) ? 1105 : 1104;
    } else {
        bw = 1101 + ((d[0] >> 5) & 0x3);
    }
    return bw;
}
CB_HD int pkt_samples_per_frame(const uint8_t *d, int Fs) {
    int a;
    if (d[0] & 0x80) {
        a = (d[0] >> 3) & 0x3;
        a = (Fs << a) / 400;
    } else if ((d[0] & 0x60) == 0x60) {
        a = (d[0] & 0x08) ? Fs / 50 : Fs / 100;
    } else {
        a = (d[0] >> 3) & 0x3;
        if (a == 3) a = Fs * 60 / 1000;
        else a = (Fs << a) / 100;
    }
    return a;
}
CB_HD int pkt_nb_channels(const uint8_t *d) { return (d[0] & 0x4) ? 2 : 1; }

CB_HD int pkt_parse_size(const uint8_t *d, int len, int16_t *size) {
    if (len < 1) { *size = -1; return -1; }
    if (d[0] < 252) { *size = d[0]; return 1; }
    if (len < 2) { *size = -1; return -1; }
    *size = (int16_t)(4 * d[1] + d[0]);
    return 2;
}

// opus_packet_parse_impl (src/opus.c:190-343).  Returns frame count or a negative error; size[48];
// *payload_offset = offset of the first frame; *packet_offset = total bytes consumed incl. padding.
CB_HD int pkt_parse(const uint8_t *data, int len, int self_delimited, uint8_t *out_toc, int16_t *size,
                    int *payload_offset, int *packet_offset) {
    int i, bytes, count, cbr = 0;
    int last_size, pad = 0;
    const uint8_t *data0 = data;
    if (size == nullptr || len < 0) return -1;
    if (len == 0) return -4;
    int framesize = pkt_samples_per_frame(data, 48000);
    uint8_t toc = *data++;
    len--;
    last_size = len;
    switch (toc & 0x3) {
    case 0:
        count = 1;
        break;
    case 1:
        count = 2;
        cbr = 1;
        if (!self_delimited) {
            if (len & 0x1) return -4;
            last_size = len / 2;
            size[0] = (int16_t)last_size;
        }
        break;
    case 2:
        count = 2;
        bytes = pkt_parse_size(data, len, size);
        len -= bytes;
        if (size[0] < 0 || size[0] > len) return -4;
        data += bytes;
        last_size = len - size[0];
        break;
    default: {
        if (len < 1) return -4;
        uint8_t ch = *data++;
        count = ch & 0x3F;
        if (count <= 0 || framesize * count > 5760) return -4;
        len--;
        if (ch & 0x40) {
            int p;
            do {
                if (len <= 0) return -4;
                p = *data++;
                len--;
                int tmp = p == 255 ? 254 : p;
                len -= tmp;
                pad += tmp;
            } while (p == 255);
        }
        if (len < 0) return -4;
        cbr = !(ch & 0x80);
        if (!cbr) {
            last_size = len;
            CB_NOUNROLL for (i = 0; i < count - 1; i++) {
                bytes = pkt_parse_size(data, len, size + i);
                len -= bytes;
                if (size[i] < 0 || size[i] > len) return -4;
                data += bytes;
                last_size -= bytes + size[i];
            }
            if (last_size < 0) return -4;
        } else if (!self_delimited) {
            last_size = len / count;
            if (last_size * count != len) return -4;
            CB_NOUNROLL for (i = 0; i < count - 1; i++) size[i] = (int16_t)last_size;
        }
        break;
    }
    }
    if (self_delimited) {
        bytes = pkt_parse_size(data, len, size + count - 1);
        len -= bytes;
        if (size[count - 1] < 0 || size[count - 1] > len) return -4;
        data += bytes;
        if (cbr) {
            if (size[count - 1] * count > len) return -4;
            CB_NOUNROLL for (i = 0; i < count - 1; i++) size[i] = size[count - 1];
        } else if (bytes + size[count - 1] > last_size) {
            return -4;
        }
    } else {
        if (last_size > 1275) return -4;
        size[count - 1] = (int16_t)last_size;
    }
    if (payload_offset) *payload_offset = (int)(data - data0);
    CB_NOUNROLL for (i = 0; i < count; i++) data += size[i];
    if (packet_offset) *packet_offset = pad + (int)(data - data0);
    if (out_toc) *out_toc = toc;
    return count;
}

// A frame length as a packet header writes it (one or two bytes; the read side is pkt_parse_size).
CB_HD int pkt_put_size(int size, uint8_t *p) {
    if (size < 252) {
        p[0] = (uint8_t)size;
        return 1;
    }
    p[0] = (uint8_t)(252 + (size & 3));
    p[1] = (uint8_t)((size - p[0]) >> 2);
    return 2;
}

// The header of an undelimited packet of `count` frames with frame-count code `code` (RFC 6716 §3.2): the TOC (configuration
// `cfg` = TOC & 0xFC), for code 2 the first frame's length, for code 3 the frame-count byte, `pad` bytes of padding as its
// length bytes (the padding itself follows the frames) and, VBR, the lengths of all frames but the last.  Returns its size
// (at most 2 + 47 * 2 + (pad + 253) / 255 bytes).
CB_HD int pkt_write_header(uint8_t *p, uint8_t cfg, int code, int count, int vbr, int pad, const int16_t *len) {
    uint8_t *q = p;
    *q++ = (uint8_t)(cfg | code);
    if (code == 2) {
        q += pkt_put_size(len[0], q);
    } else if (code == 3) {
        *q++ = (uint8_t)(count | (vbr ? 0x80 : 0) | (pad ? 0x40 : 0));
        if (pad) {
            const int n255 = (pad - 1) / 255;
            for (int i = 0; i < n255; i++) *q++ = 255;
            *q++ = (uint8_t)(pad - 255 * n255 - 1);
        }
        if (vbr)
            for (int i = 0; i < count - 1; i++) q += pkt_put_size(len[i], q);
    }
    return (int)(q - p);
}

// How `count` frames of lengths len[] are laid out by opus_repacketizer_out_range_impl (repacketizer.c:102-227): the cheapest code
// that can carry them (0: one frame, 1: two equal, 2: two different, 3: any count, CBR or VBR) — code 3 is forced when padding is
// wanted and there is room for it.  `sd` is the size of a self-delimiting length (0 for an ordinary packet, else 1 or 2 bytes for
// the last frame's length), which counts towards header and total.  Returns 0 or OPUS_BUFFER_TOO_SMALL when the packet exceeds
// maxlen; with want_pad the packet is padded to exactly maxlen (pad includes the padding-length bytes themselves).
struct PktLayout {
    int code, vbr, header, total, pad;
};
CB_HD int plan_layout(const int16_t *len, int count, int maxlen, int want_pad, PktLayout &L, int sd = 0) {
    int payload = 0;
    for (int i = 0; i < count; i++) payload += len[i];
    L.pad = 0;
    L.vbr = 0;
    if (count == 1) { L.code = 0; L.header = 1; }
    else if (count == 2 && len[0] == len[1]) { L.code = 1; L.header = 1; }
    else if (count == 2) { L.code = 2; L.header = 1 + 1 + (len[0] >= 252); }
    else L.code = 3;
    if (L.code != 3) {
        L.header += sd;
        L.total = L.header + payload;
        if (L.total > maxlen) return -2;   // OPUS_BUFFER_TOO_SMALL
        if (!(want_pad && L.total < maxlen)) return 0;
        L.code = 3;   // padding needs the code-3 header
    }
    for (int i = 1; i < count; i++)
        if (len[i] != len[0]) { L.vbr = 1; break; }
    L.header = 2 + sd;
    if (L.vbr)
        for (int i = 0; i < count - 1; i++) L.header += 1 + (len[i] >= 252);
    L.total = L.header + payload;
    if (L.total > maxlen) return -2;
    if (want_pad && L.total < maxlen) {
        L.pad = maxlen - L.total;
        L.total = maxlen;
    }
    return 0;
}

}  // namespace cb

// opus_repacketizer.cu — host half of the C ABI that only moves bytes: the repacketizer and opus_packet_pad / opus_packet_unpad
// for any packet (frame-count codes 0-3).  Interface: opus-fix/include/opus.h:628-750, behaviour: src/repacketizer.c:37-273
// (same return codes, same byte layout of the packets it writes).  No device code: packets are parsed with csrc/opus_packet.h,
// the parser the decoder kernels use.
#include <cstdlib>
#include <cstring>

#include "../../include/opus_b200.h"
#include "celt_simt.cuh"
#include "opus_packet.h"

// Frames collected by opus_repacketizer_cat.  The frames point into the caller's packets (opus.h: "the repacketizer state contains
// pointers to the submitted packets"), so those must stay valid until the next init.
struct OpusRepacketizer {
    unsigned char toc;
    int nb_frames;
    const unsigned char *frames[48];
    opus_int16 len[48];
    int framesize;   // samples per frame at 8 kHz: 120 ms = 960
};

namespace {

// opus_repacketizer_out_range_impl (repacketizer.c:102-227) without self-delimited framing.  `data` may overlap the frames as
// long as every frame lies at or after the place it is moved to (in-place pad / unpad): frames are moved front to back.
opus_int32 emit_range(const OpusRepacketizer *rp, int begin, int end, unsigned char *data, opus_int32 maxlen, int want_pad) {
    if (begin < 0 || begin >= end || end > rp->nb_frames) return OPUS_BAD_ARG;
    const int count = end - begin;
    const opus_int16 *len = rp->len + begin;
    const unsigned char *const *frames = rp->frames + begin;
    cb::PktLayout L;
    const int rc = cb::plan_layout(len, count, maxlen, want_pad, L);
    if (rc != OPUS_OK) return rc;
    unsigned char *p = data;
    p += cb::pkt_write_header(p, (unsigned char)(rp->toc & 0xFC), L.code, count, L.vbr, L.pad, len);
    for (int i = 0; i < count; i++) {
        memmove(p, frames[i], (size_t)len[i]);
        p += len[i];
    }
    if (want_pad)
        while (p < data + maxlen) *p++ = 0;
    return L.total;
}

}  // namespace

extern "C" {

int opus_repacketizer_get_size(void) { return (int)sizeof(OpusRepacketizer); }

OpusRepacketizer *opus_repacketizer_init(OpusRepacketizer *rp) {
    rp->nb_frames = 0;
    return rp;
}

OpusRepacketizer *opus_repacketizer_create(void) {
    OpusRepacketizer *rp = (OpusRepacketizer *)malloc(sizeof(OpusRepacketizer));
    return rp ? opus_repacketizer_init(rp) : nullptr;
}

void opus_repacketizer_destroy(OpusRepacketizer *rp) { free(rp); }

// repacketizer.c:62-97
int opus_repacketizer_cat(OpusRepacketizer *rp, const unsigned char *data, opus_int32 len) {
    if (len < 1) return OPUS_INVALID_PACKET;
    if (rp->nb_frames == 0) {
        rp->toc = data[0];
        rp->framesize = cb::pkt_samples_per_frame(data, 8000);
    } else if ((rp->toc & 0xFC) != (data[0] & 0xFC)) {
        return OPUS_INVALID_PACKET;
    }
    const int incoming = opus_packet_get_nb_frames(data, len);
    if (incoming < 1) return OPUS_INVALID_PACKET;
    if ((incoming + rp->nb_frames) * rp->framesize > 960) return OPUS_INVALID_PACKET;   // 120 ms at most
    unsigned char toc;
    int offset = 0;
    const int n = cb::pkt_parse(data, len, 0, &toc, rp->len + rp->nb_frames, &offset, nullptr);
    if (n < 1) return n;
    const unsigned char *p = data + offset;
    for (int i = 0; i < n; i++) {
        rp->frames[rp->nb_frames + i] = p;
        p += rp->len[rp->nb_frames + i];
    }
    rp->nb_frames += incoming;
    return OPUS_OK;
}

int opus_repacketizer_get_nb_frames(OpusRepacketizer *rp) { return rp->nb_frames; }

opus_int32 opus_repacketizer_out_range(OpusRepacketizer *rp, int begin, int end, unsigned char *data, opus_int32 maxlen) {
    return emit_range(rp, begin, end, data, maxlen, 0);
}

opus_int32 opus_repacketizer_out(OpusRepacketizer *rp, unsigned char *data, opus_int32 maxlen) {
    return emit_range(rp, 0, rp->nb_frames, data, maxlen, 0);
}

// repacketizer.c:239-258: the packet is first moved to the end of the buffer, then re-emitted at its start with padding
int opus_packet_pad(unsigned char *data, opus_int32 len, opus_int32 new_len) {
    if (len < 1) return OPUS_BAD_ARG;
    if (len == new_len) return OPUS_OK;
    if (len > new_len) return OPUS_BAD_ARG;
    OpusRepacketizer rp;
    opus_repacketizer_init(&rp);
    memmove(data + new_len - len, data, (size_t)len);
    opus_repacketizer_cat(&rp, data + new_len - len, len);
    const opus_int32 ret = emit_range(&rp, 0, rp.nb_frames, data, new_len, 1);
    return ret > 0 ? OPUS_OK : ret;
}

// repacketizer.c:260-273
opus_int32 opus_packet_unpad(unsigned char *data, opus_int32 len) {
    if (len < 1) return OPUS_BAD_ARG;
    OpusRepacketizer rp;
    opus_repacketizer_init(&rp);
    const int rc = opus_repacketizer_cat(&rp, data, len);
    if (rc < 0) return rc;
    return emit_range(&rp, 0, rp.nb_frames, data, len, 0);
}

}  // extern "C"

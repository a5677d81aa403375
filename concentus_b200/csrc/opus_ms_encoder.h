// opus_ms_encoder.h — the multistream encoder's layout, rate allocation and byte budgets, usable from host and device code.
//
// A restatement of libopus 1.1.x src/opus_multistream_encoder.c (validate_encoder_layout, opus_multistream_surround_encoder_init,
// surround_rate_allocation, opus_multistream_encode_native) for the scope this library builds: no surround analysis, no LFE
// stream, 16-bit input.  The host C ABI (opus_enc_capi.cu), its kernels and the host-simulation tests all call these functions.
//
// Readings taken where libopus versions differ (none of them has been checked against a reference build):
//  - a call with max_data_bytes < 4·S − 1 is OPUS_BUFFER_TOO_SMALL (ms_enc_min_bytes);
//  - the stream offset includes 60·(Fs/frame_size − 50) (ms_rate_allocation);
//  - CBR caps max_data_bytes at 3·B / (3·8·Fs/frame_size) with B as stored, OPUS_AUTO and OPUS_BITRATE_MAX included
//    (ms_cbr_max_bytes);
//  - stream s's budget reserves max(0, 4·(S−s−1) − 1) bytes for the streams after it and is at most 3·1275 + 7 bytes
//    (ms_stream_budget), with no further reservation for its self-delimiting length;
//  - OPUS_SET_BITRATE on the multistream encoder stores any value ≥ 0, OPUS_AUTO or OPUS_BITRATE_MAX without clamping.
#pragma once
#include <stdint.h>
#include "opus_packet.h"

namespace cb {

enum { kMsFrameTmp = 3 * 1275 + 7 };   // MS_FRAME_TMP: the most one stream may be given

// The first input channel that carries stream channel `k` (get_left/right/mono_channel with prev = -1), or -1.
CB_HD int ms_enc_source_channel(const uint8_t *mapping, int channels, int k) {
    for (int c = 0; c < channels; c++)
        if (mapping[c] == k) return c;
    return -1;
}

// opus_multistream_encoder_init's argument and layout rules (validate_layout, validate_encoder_layout): 0 or OPUS_BAD_ARG.
CB_HD int ms_enc_check_layout(int channels, int streams, int coupled, const uint8_t *mapping) {
    if (channels > 255 || channels < 1 || coupled > streams || streams < 1 || coupled < 0 || streams > 255 - coupled) return -1;
    for (int c = 0; c < channels; c++)
        if (mapping[c] >= streams + coupled && mapping[c] != 255) return -1;
    for (int s = 0; s < streams; s++) {
        if (s < coupled) {
            if (ms_enc_source_channel(mapping, channels, 2 * s) < 0 || ms_enc_source_channel(mapping, channels, 2 * s + 1) < 0) return -1;
        } else if (ms_enc_source_channel(mapping, channels, coupled + s) < 0) {
            return -1;
        }
    }
    return 0;
}

// The layout opus_multistream_surround_encoder_init chooses, for the families this library builds: family 0 with 1 or 2
// channels, family 1 with 1 or 2 channels (the Vorbis order of RFC 7845 §5.1.1.2), family 255 (one mono stream per channel).
// Family 1 with 3-8 channels needs surround masking and an LFE stream: OPUS_UNIMPLEMENTED, like every other family.
// Returns 0, OPUS_BAD_ARG (channels outside 1..255) or OPUS_UNIMPLEMENTED.
CB_HD int ms_surround_layout(int channels, int family, int *streams, int *coupled, uint8_t *mapping) {
    if (channels > 255 || channels < 1) return -1;
    if ((family == 0 || family == 1) && channels <= 2) {
        *streams = 1;
        *coupled = channels - 1;
        for (int c = 0; c < channels; c++) mapping[c] = (uint8_t)c;
        return 0;
    }
    if (family == 255) {
        *streams = channels;
        *coupled = 0;
        for (int c = 0; c < channels; c++) mapping[c] = (uint8_t)c;
        return 0;
    }
    return -5;
}

// opus_multistream_encode_native's first size check: the smallest packet that can carry S streams.
CB_HD int ms_enc_min_bytes(int streams) { return 4 * streams - 1; }

// surround_rate_allocation with no LFE stream: the bitrate each stream is set to for one call, from the multistream bitrate B
// (OPUS_AUTO = -1000, OPUS_BITRATE_MAX = -1, else as stored) of a C-channel encoder.  C integer semantics (truncating division);
// the product 256·(B − offset·S) is formed in 64 bits and each rate saturates at INT32_MAX, where the reference's int arithmetic
// would overflow (B above about 8 Mbit/s).
CB_HD void ms_rate_allocation(int B, int channels, int streams, int coupled, int Fs, int frame_size, int32_t *rate) {
    int stream_offset = B > 40000 * channels ? 20000 : B / channels / 2;
    stream_offset += 60 * (Fs / frame_size - 50);
    int64_t channel_rate;
    if (B == -1000) channel_rate = Fs + 60 * Fs / frame_size;
    else if (B == -1) channel_rate = 300000;
    else channel_rate = 256 * ((int64_t)B - (int64_t)stream_offset * streams) / (256 * (streams - coupled) + 512 * coupled);
    for (int s = 0; s < streams; s++) {
        int64_t r = stream_offset + (s < coupled ? (channel_rate * 512) >> 8 : channel_rate);
        rate[s] = (int32_t)(r > 2147483647 ? 2147483647 : (r < -2147483647 - 1 ? -2147483647 - 1 : r));
    }
}

// CBR: max_data_bytes = min(max_data_bytes, 3·B / (3·8·Fs/frame_size)), B as stored.
CB_HD int ms_cbr_max_bytes(int max_data_bytes, int B, int Fs, int frame_size) {
    const int cap = 3 * B / (3 * 8 * Fs / frame_size);
    return max_data_bytes < cap ? max_data_bytes : cap;
}

// The byte budget of stream s of S once the streams before it took tot_size bytes of a packet of max_data_bytes.
CB_HD int ms_stream_budget(int max_data_bytes, int tot_size, int streams, int s) {
    int curr_max = max_data_bytes - tot_size;
    const int reserve = 4 * (streams - s - 1) - 1;
    curr_max -= reserve > 0 ? reserve : 0;
    return curr_max < kMsFrameTmp ? curr_max : kMsFrameTmp;
}

// CBR: the bitrate the last stream is set to before it is coded, from its budget.
CB_HD int ms_cbr_last_bitrate(int curr_max, int Fs, int frame_size) { return curr_max * (8 * Fs / frame_size); }

}  // namespace cb

/* opus_b200.h — C ABI of libconcentus_b200.so: a drop-in for the CELT frame path of libopus 1.1.2
 * (opus-fix FIXED_POINT build), executed by hand-written sm_100a CUDA kernels.
 *
 * Every entry point below is `extern "C"`, takes plain pointers and sizes, and has exactly the name,
 * argument meaning and return convention of the reference function it replaces (file:line cited).
 * The batch / span entry points at the end are ours (SURVEY.md §8b): semantically a loop of the scalar
 * call over independent streams, executed as one kernel launch with one warp per stream.
 *
 * Scope edge (SURVEY.md §8b): only MODE_CELT_ONLY packets (TOC bit 7 set) are decoded; SILK-only / hybrid
 * packets return OPUS_UNIMPLEMENTED and leave the state untouched.  There is no CPU fallback: every
 * codec call fails with OPUS_INTERNAL_ERROR if no CUDA device is usable.
 */
#ifndef OPUS_B200_H
#define OPUS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef int32_t opus_int32;
typedef uint32_t opus_uint32;
typedef int16_t opus_int16;

/* Error codes — opus-fix/include/opus_defines.h:46-60 */
#define OPUS_OK 0
#define OPUS_BAD_ARG -1
#define OPUS_BUFFER_TOO_SMALL -2
#define OPUS_INTERNAL_ERROR -3
#define OPUS_INVALID_PACKET -4
#define OPUS_UNIMPLEMENTED -5
#define OPUS_INVALID_STATE -6
#define OPUS_ALLOC_FAIL -7

/* ctl request numbers — opus-fix/include/opus_defines.h:130-167 */
#define OPUS_SET_APPLICATION_REQUEST 4000
#define OPUS_GET_APPLICATION_REQUEST 4001
#define OPUS_SET_BITRATE_REQUEST 4002
#define OPUS_GET_BITRATE_REQUEST 4003
#define OPUS_SET_MAX_BANDWIDTH_REQUEST 4004
#define OPUS_GET_MAX_BANDWIDTH_REQUEST 4005
#define OPUS_SET_VBR_REQUEST 4006
#define OPUS_GET_VBR_REQUEST 4007
#define OPUS_SET_BANDWIDTH_REQUEST 4008
#define OPUS_GET_BANDWIDTH_REQUEST 4009
#define OPUS_SET_COMPLEXITY_REQUEST 4010
#define OPUS_GET_COMPLEXITY_REQUEST 4011
#define OPUS_SET_INBAND_FEC_REQUEST 4012
#define OPUS_GET_INBAND_FEC_REQUEST 4013
#define OPUS_SET_PACKET_LOSS_PERC_REQUEST 4014
#define OPUS_GET_PACKET_LOSS_PERC_REQUEST 4015
#define OPUS_SET_DTX_REQUEST 4016
#define OPUS_GET_DTX_REQUEST 4017
#define OPUS_SET_VBR_CONSTRAINT_REQUEST 4020
#define OPUS_GET_VBR_CONSTRAINT_REQUEST 4021
#define OPUS_SET_FORCE_CHANNELS_REQUEST 4022
#define OPUS_GET_FORCE_CHANNELS_REQUEST 4023
#define OPUS_SET_SIGNAL_REQUEST 4024
#define OPUS_GET_SIGNAL_REQUEST 4025
#define OPUS_GET_LOOKAHEAD_REQUEST 4027
#define OPUS_RESET_STATE 4028
#define OPUS_GET_SAMPLE_RATE_REQUEST 4029
#define OPUS_GET_FINAL_RANGE_REQUEST 4031
#define OPUS_GET_PITCH_REQUEST 4033
#define OPUS_SET_GAIN_REQUEST 4034
#define OPUS_GET_GAIN_REQUEST 4045
#define OPUS_SET_LSB_DEPTH_REQUEST 4036
#define OPUS_GET_LSB_DEPTH_REQUEST 4037
#define OPUS_GET_LAST_PACKET_DURATION_REQUEST 4039
#define OPUS_SET_EXPERT_FRAME_DURATION_REQUEST 4040
#define OPUS_GET_EXPERT_FRAME_DURATION_REQUEST 4041
#define OPUS_SET_PREDICTION_DISABLED_REQUEST 4042
#define OPUS_GET_PREDICTION_DISABLED_REQUEST 4043
#define OPUS_SET_FORCE_MODE_REQUEST 11002 /* opus-fix/src/opus_private.h */

/* The reference's argument-checked convenience macros (opus-fix/include/opus_defines.h:107-122,260-660; celt/celt.h:113-117), so
 * that sources written against opus.h — opus_encoder_ctl(enc, OPUS_SET_BITRATE(64000)) — compile against this header unchanged. */
#define __opus_check_int(x) (((void)((x) == (opus_int32)0)), (opus_int32)(x))
#define __opus_check_int_ptr(ptr) ((ptr) + ((ptr) - (opus_int32 *)(ptr)))
#define __opus_check_uint_ptr(ptr) ((ptr) + ((ptr) - (opus_uint32 *)(ptr)))
#define OPUS_SET_APPLICATION(x) OPUS_SET_APPLICATION_REQUEST, __opus_check_int(x)
#define OPUS_GET_APPLICATION(x) OPUS_GET_APPLICATION_REQUEST, __opus_check_int_ptr(x)
#define OPUS_SET_BITRATE(x) OPUS_SET_BITRATE_REQUEST, __opus_check_int(x)
#define OPUS_GET_BITRATE(x) OPUS_GET_BITRATE_REQUEST, __opus_check_int_ptr(x)
#define OPUS_SET_MAX_BANDWIDTH(x) OPUS_SET_MAX_BANDWIDTH_REQUEST, __opus_check_int(x)
#define OPUS_GET_MAX_BANDWIDTH(x) OPUS_GET_MAX_BANDWIDTH_REQUEST, __opus_check_int_ptr(x)
#define OPUS_SET_VBR(x) OPUS_SET_VBR_REQUEST, __opus_check_int(x)
#define OPUS_GET_VBR(x) OPUS_GET_VBR_REQUEST, __opus_check_int_ptr(x)
#define OPUS_SET_BANDWIDTH(x) OPUS_SET_BANDWIDTH_REQUEST, __opus_check_int(x)
#define OPUS_GET_BANDWIDTH(x) OPUS_GET_BANDWIDTH_REQUEST, __opus_check_int_ptr(x)
#define OPUS_SET_COMPLEXITY(x) OPUS_SET_COMPLEXITY_REQUEST, __opus_check_int(x)
#define OPUS_GET_COMPLEXITY(x) OPUS_GET_COMPLEXITY_REQUEST, __opus_check_int_ptr(x)
#define OPUS_SET_INBAND_FEC(x) OPUS_SET_INBAND_FEC_REQUEST, __opus_check_int(x)
#define OPUS_GET_INBAND_FEC(x) OPUS_GET_INBAND_FEC_REQUEST, __opus_check_int_ptr(x)
#define OPUS_SET_PACKET_LOSS_PERC(x) OPUS_SET_PACKET_LOSS_PERC_REQUEST, __opus_check_int(x)
#define OPUS_GET_PACKET_LOSS_PERC(x) OPUS_GET_PACKET_LOSS_PERC_REQUEST, __opus_check_int_ptr(x)
#define OPUS_SET_DTX(x) OPUS_SET_DTX_REQUEST, __opus_check_int(x)
#define OPUS_GET_DTX(x) OPUS_GET_DTX_REQUEST, __opus_check_int_ptr(x)
#define OPUS_SET_VBR_CONSTRAINT(x) OPUS_SET_VBR_CONSTRAINT_REQUEST, __opus_check_int(x)
#define OPUS_GET_VBR_CONSTRAINT(x) OPUS_GET_VBR_CONSTRAINT_REQUEST, __opus_check_int_ptr(x)
#define OPUS_SET_FORCE_CHANNELS(x) OPUS_SET_FORCE_CHANNELS_REQUEST, __opus_check_int(x)
#define OPUS_GET_FORCE_CHANNELS(x) OPUS_GET_FORCE_CHANNELS_REQUEST, __opus_check_int_ptr(x)
#define OPUS_SET_SIGNAL(x) OPUS_SET_SIGNAL_REQUEST, __opus_check_int(x)
#define OPUS_GET_SIGNAL(x) OPUS_GET_SIGNAL_REQUEST, __opus_check_int_ptr(x)
#define OPUS_GET_LOOKAHEAD(x) OPUS_GET_LOOKAHEAD_REQUEST, __opus_check_int_ptr(x)
#define OPUS_GET_SAMPLE_RATE(x) OPUS_GET_SAMPLE_RATE_REQUEST, __opus_check_int_ptr(x)
#define OPUS_GET_FINAL_RANGE(x) OPUS_GET_FINAL_RANGE_REQUEST, __opus_check_uint_ptr(x)
#define OPUS_GET_PITCH(x) OPUS_GET_PITCH_REQUEST, __opus_check_int_ptr(x)
#define OPUS_SET_GAIN(x) OPUS_SET_GAIN_REQUEST, __opus_check_int(x)
#define OPUS_GET_GAIN(x) OPUS_GET_GAIN_REQUEST, __opus_check_int_ptr(x)
#define OPUS_SET_LSB_DEPTH(x) OPUS_SET_LSB_DEPTH_REQUEST, __opus_check_int(x)
#define OPUS_GET_LSB_DEPTH(x) OPUS_GET_LSB_DEPTH_REQUEST, __opus_check_int_ptr(x)
#define OPUS_GET_LAST_PACKET_DURATION(x) OPUS_GET_LAST_PACKET_DURATION_REQUEST, __opus_check_int_ptr(x)
#define OPUS_SET_EXPERT_FRAME_DURATION(x) OPUS_SET_EXPERT_FRAME_DURATION_REQUEST, __opus_check_int(x)
#define OPUS_GET_EXPERT_FRAME_DURATION(x) OPUS_GET_EXPERT_FRAME_DURATION_REQUEST, __opus_check_int_ptr(x)
#define OPUS_SET_PREDICTION_DISABLED(x) OPUS_SET_PREDICTION_DISABLED_REQUEST, __opus_check_int(x)
#define OPUS_GET_PREDICTION_DISABLED(x) OPUS_GET_PREDICTION_DISABLED_REQUEST, __opus_check_int_ptr(x)
#define OPUS_SET_FORCE_MODE(x) OPUS_SET_FORCE_MODE_REQUEST, __opus_check_int(x)
/* multistream-only switches of the CELT layer: only their defaults are accepted (DESIGN.md 6) */
#define OPUS_SET_LFE_REQUEST 10024
#define OPUS_SET_LFE(x) OPUS_SET_LFE_REQUEST, __opus_check_int(x)
#define OPUS_SET_ENERGY_MASK_REQUEST 10026
#define OPUS_SET_ENERGY_MASK(x) OPUS_SET_ENERGY_MASK_REQUEST, (x)

#define OPUS_AUTO -1000
#define OPUS_BITRATE_MAX -1
#define OPUS_APPLICATION_VOIP 2048
#define OPUS_APPLICATION_AUDIO 2049
#define OPUS_APPLICATION_RESTRICTED_LOWDELAY 2051
#define OPUS_BANDWIDTH_NARROWBAND 1101
#define OPUS_BANDWIDTH_MEDIUMBAND 1102
#define OPUS_BANDWIDTH_WIDEBAND 1103
#define OPUS_BANDWIDTH_SUPERWIDEBAND 1104
#define OPUS_BANDWIDTH_FULLBAND 1105

typedef struct OpusDecoder OpusDecoder;
typedef struct OpusEncoder OpusEncoder;

/* ---- decoder: opus-fix/include/opus.h:406-512, src/opus_decoder.c:82-166,713-719,802-919 ---- */
int opus_decoder_get_size(int channels);                                            /* opus_decoder.c:82  */
OpusDecoder *opus_decoder_create(opus_int32 Fs, int channels, int *error);          /* opus_decoder.c:139 */
int opus_decoder_init(OpusDecoder *st, opus_int32 Fs, int channels);                /* opus_decoder.c:96  */
int opus_decode(OpusDecoder *st, const unsigned char *data, opus_int32 len, opus_int16 *pcm, int frame_size,
                int decode_fec);                                                    /* opus_decoder.c:713 */
int opus_decoder_ctl(OpusDecoder *st, int request, ...);                            /* opus_decoder.c:802 */
void opus_decoder_destroy(OpusDecoder *st);                                         /* opus_decoder.c:915 */

/* ---- encoder: opus-fix/include/opus.h:171-328, src/opus_encoder.c:150-252,482-510,2007-2507 ----
 * Scope (SURVEY.md section 8b): frames are coded in MODE_CELT_ONLY (OPUS_APPLICATION_RESTRICTED_LOWDELAY, or
 * OPUS_APPLICATION_AUDIO when the reference's own mode decision / OPUS_SET_FORCE_MODE picks CELT), 8-48 kHz, 2.5-60 ms.
 * A frame the reference would code with SILK/hybrid and OPUS_APPLICATION_VOIP return
 * OPUS_UNIMPLEMENTED and leave the state untouched. */
int opus_encoder_get_size(int channels);                                                        /* opus_encoder.c:150 */
OpusEncoder *opus_encoder_create(opus_int32 Fs, int channels, int application, int *error);     /* opus_encoder.c:482 */
int opus_encoder_init(OpusEncoder *st, opus_int32 Fs, int channels, int application);           /* opus_encoder.c:164 */
opus_int32 opus_encode(OpusEncoder *st, const opus_int16 *pcm, int frame_size, unsigned char *data,
                       opus_int32 max_data_bytes);                                              /* opus_encoder.c:2007 */
int opus_encoder_ctl(OpusEncoder *st, int request, ...);                                        /* opus_encoder.c:2031 */
void opus_encoder_destroy(OpusEncoder *st);                                                     /* opus_encoder.c:2509 */
int opus_packet_pad(unsigned char *data, opus_int32 len, opus_int32 new_len);                   /* repacketizer.c:239 */
opus_int32 opus_packet_unpad(unsigned char *data, opus_int32 len);                              /* repacketizer.c:260 */

/* ---- repacketizer: opus-fix/include/opus.h:628-750, src/repacketizer.c:37-236 (host code: merges / splits packets of one
 * configuration without touching the compressed frames) ---- */
typedef struct OpusRepacketizer OpusRepacketizer;
int opus_repacketizer_get_size(void);                                                           /* repacketizer.c:37  */
OpusRepacketizer *opus_repacketizer_init(OpusRepacketizer *rp);                                 /* repacketizer.c:42  */
OpusRepacketizer *opus_repacketizer_create(void);                                               /* repacketizer.c:48  */
void opus_repacketizer_destroy(OpusRepacketizer *rp);                                           /* repacketizer.c:57  */
int opus_repacketizer_cat(OpusRepacketizer *rp, const unsigned char *data, opus_int32 len);     /* repacketizer.c:93  */
int opus_repacketizer_get_nb_frames(OpusRepacketizer *rp);                                      /* repacketizer.c:98  */
opus_int32 opus_repacketizer_out_range(OpusRepacketizer *rp, int begin, int end, unsigned char *data,
                                       opus_int32 maxlen);                                      /* repacketizer.c:229 */
opus_int32 opus_repacketizer_out(OpusRepacketizer *rp, unsigned char *data, opus_int32 maxlen); /* repacketizer.c:234 */

/* ---- packet helpers: opus-fix/include/opus.h:527-594, src/opus.c:169-352, src/opus_decoder.c:921-981 ---- */
int opus_packet_parse(const unsigned char *data, opus_int32 len, unsigned char *out_toc, const unsigned char *frames[48],
                      opus_int16 size[48], int *payload_offset);
int opus_packet_get_bandwidth(const unsigned char *data);
int opus_packet_get_samples_per_frame(const unsigned char *data, opus_int32 Fs);
int opus_packet_get_nb_channels(const unsigned char *data);
int opus_packet_get_nb_frames(const unsigned char packet[], opus_int32 len);
int opus_packet_get_nb_samples(const unsigned char packet[], opus_int32 len, opus_int32 Fs);
int opus_decoder_get_nb_samples(const OpusDecoder *dec, const unsigned char packet[], opus_int32 len);
const char *opus_strerror(int error);                                               /* celt/celt.c:268-284 */
const char *opus_get_version_string(void);                                          /* celt/celt.c:286-299 */

/* ---- batch entry points (ours).  ret[i] is what the scalar call on stream i would have returned. ---- */

/* One packet for each of n independent streams.  Semantics: for i in 0..n-1: ret[i] = opus_decode(st[i], data[i],
 * len[i], pcm[i], frame_size, decode_fec).  Host buffers.  The states stay resident in HBM afterwards; any scalar
 * call / ctl on them, or opus_decoder_sync(), writes them back into the caller's blocks first. */
int opus_decode_batch(OpusDecoder **st, const unsigned char *const *data, const opus_int32 *len, opus_int16 *const *pcm,
                      int frame_size, int decode_fec, int *ret, int n);

/* A span of F consecutive packets for each of n streams, one launch.  Packet (s,f) occupies
 * data[offs[s*F+f] .. +len[s*F+f]); its PCM goes to pcm + (s*F+f)*frame_size*channels (frame_size = capacity
 * per packet, samples per channel); ret[s*F+f] as above.  All streams must share Fs and channel count.
 * Host buffers: copies to/from the device are part of the call. */
int opus_decode_span(OpusDecoder **st, int n, int F, const unsigned char *data, const int64_t *offs, const opus_int32 *len,
                     opus_int16 *pcm, int frame_size, int *ret);

/* Same, but data/offs/len/pcm/ret are DEVICE pointers (inputs already resident in HBM) and the call only
 * enqueues the kernel on the library's stream; opus_b200_synchronize() waits for it. */
int opus_decode_span_device(OpusDecoder **st, int n, int F, const unsigned char *d_data, const int64_t *d_offs,
                            const opus_int32 *d_len, opus_int16 *d_pcm, int frame_size, int *d_ret);

/* Write device-resident states back into the caller-visible blocks (memcpy-able again) and release residency. */
int opus_decoder_sync(OpusDecoder **st, int n);

/* Encoder counterparts.  opus_encode_batch: for i in 0..n-1: ret[i] = opus_encode(st[i], pcm[i], frame_size, data[i],
 * max_data_bytes).  opus_encode_span: F consecutive frames for each of n streams in one launch; PCM of frame (s,f) is
 * pcm + (s*F+f)*frame_size*channels, its packet is written at data + (s*F+f)*max_data_bytes (max_data_bytes is both the
 * size limit of a packet, clamped to 1276 like opus_encoder.c:980, and the slot stride), ret[s*F+f] = packet length or
 * error.  All streams of a span must share Fs and channel count.  _device: pcm/data/ret are DEVICE pointers, the call only
 * enqueues; opus_b200_enc_synchronize() waits. */
int opus_encode_batch(OpusEncoder **st, const opus_int16 *const *pcm, int frame_size, unsigned char *const *data,
                      opus_int32 max_data_bytes, opus_int32 *ret, int n);
int opus_encode_span(OpusEncoder **st, int n, int F, const opus_int16 *pcm, int frame_size, unsigned char *data,
                     opus_int32 max_data_bytes, opus_int32 *ret);
int opus_encode_span_device(OpusEncoder **st, int n, int F, const opus_int16 *d_pcm, int frame_size, unsigned char *d_data,
                            opus_int32 max_data_bytes, opus_int32 *d_ret);
/* opus_encode_span that also reports OPUS_GET_FINAL_RANGE after every frame: final_range[s*F+f] — what opus_demo stores next to
 * each packet in its .bit container (src/opus_demo.c:748-760) and checks against its decoder (:806-816). */
int opus_encode_span_ranges(OpusEncoder **st, int n, int F, const opus_int16 *pcm, int frame_size, unsigned char *data,
                            opus_int32 max_data_bytes, opus_int32 *ret, opus_uint32 *final_range);
int opus_encoder_sync(OpusEncoder **st, int n);

/* ---- multistream decoder: libopus opus_multistream.h (opus_multistream_decoder_*), packet format RFC 6716 Appendix B, channel
 * mapping RFC 7845 section 5.1.1.  `streams` Opus streams, the first `coupled_streams` stereo and the rest mono; coupled stream s
 * decodes stream channels 2s and 2s+1, mono stream s stream channel coupled_streams + s; output channel c is a copy of stream channel
 * mapping[c], or silence when mapping[c] == 255.  Streams 0..streams-2 of a packet are self-delimited, the last one takes the
 * remaining bytes.  A packet is validated whole before any stream is decoded, so a rejected packet leaves every stream untouched;
 * a SILK or hybrid sub-packet that carries a frame is OPUS_UNIMPLEMENTED like in opus_decode. ---- */
typedef struct OpusMSDecoder OpusMSDecoder;
#define OPUS_MULTISTREAM_GET_DECODER_STATE_REQUEST 5122
#define __opus_check_decstate_ptr(ptr) ((ptr) + ((ptr) - (OpusDecoder **)(ptr)))
#define OPUS_MULTISTREAM_GET_DECODER_STATE(x, y) OPUS_MULTISTREAM_GET_DECODER_STATE_REQUEST, __opus_check_int(x), __opus_check_decstate_ptr(y)
opus_int32 opus_multistream_decoder_get_size(int streams, int coupled_streams);
OpusMSDecoder *opus_multistream_decoder_create(opus_int32 Fs, int channels, int streams, int coupled_streams, const unsigned char *mapping,
                                               int *error);
int opus_multistream_decoder_init(OpusMSDecoder *st, opus_int32 Fs, int channels, int streams, int coupled_streams,
                                  const unsigned char *mapping);
int opus_multistream_decode(OpusMSDecoder *st, const unsigned char *data, opus_int32 len, opus_int16 *pcm, int frame_size, int decode_fec);
/* OPUS_RESET_STATE and OPUS_SET_GAIN go to every stream; OPUS_GET_BANDWIDTH, _SAMPLE_RATE, _GAIN and _LAST_PACKET_DURATION are
 * answered by stream 0; OPUS_GET_FINAL_RANGE is the XOR of all streams' final ranges; OPUS_MULTISTREAM_GET_DECODER_STATE(id, &dec)
 * gives the embedded OpusDecoder of stream id, on which opus_decoder_ctl works. */
int opus_multistream_decoder_ctl(OpusMSDecoder *st, int request, ...);
void opus_multistream_decoder_destroy(OpusMSDecoder *st);

/* Multistream spans (ours), the contracts of opus_decode_span / _span_device / opus_decoder_sync: multistream packet (m,f) at
 * data[offs[m*F+f] .. +len[m*F+f]), its PCM at pcm + (m*F+f)*frame_size*channels, ret[m*F+f] what opus_multistream_decode returns.
 * Every decoder of a span shares Fs, channels, streams and coupled_streams; mappings may differ.  Packets that overlap must do so
 * whole (the same bytes at the same offset). */
int opus_multistream_decode_span(OpusMSDecoder **st, int n, int F, const unsigned char *data, const int64_t *offs, const opus_int32 *len,
                                 opus_int16 *pcm, int frame_size, int *ret);
int opus_multistream_decode_span_device(OpusMSDecoder **st, int n, int F, const unsigned char *d_data, const int64_t *d_offs,
                                        const opus_int32 *d_len, opus_int16 *d_pcm, int frame_size, int *d_ret);
int opus_multistream_decoder_sync(OpusMSDecoder **st, int n);

/* ---- multistream encoder: libopus opus_multistream.h (opus_multistream_encoder_*, opus_multistream_surround_encoder_*), the
 * packet format of the multistream decoder above.  Input channel c feeds stream channel mapping[c] (255: the channel is ignored);
 * a stream channel fed by several input channels takes the first of them.  Every coupled stream needs both of its channels and
 * every mono stream its channel, else init is OPUS_BAD_ARG.  Each call gives every stream its share of the multistream bitrate
 * (libopus's surround_rate_allocation without an LFE stream) and codes the streams in order, each within the bytes the earlier
 * ones left (at most 1276 per stream, the single-stream clamp of opus_encode); in CBR the last stream is padded to fill the packet.
 * A stream that fails ends the call with its error: the streams before it have advanced, those after it are untouched.
 * Surround masking and LFE streams are not built: the surround encoder takes mapping families 0 and 1 with 1-2 channels and
 * family 255, and returns OPUS_UNIMPLEMENTED for family 1 with 3-8 channels.  A 5.1 stream can still be written with the explicit
 * layout (streams 4, coupled 2, mapping {0,4,1,2,3,5}); it is a valid family-1 stream, not the one libopus's surround encoder
 * would write. ---- */
typedef struct OpusMSEncoder OpusMSEncoder;
#define OPUS_MULTISTREAM_GET_ENCODER_STATE_REQUEST 5120
#define __opus_check_encstate_ptr(ptr) ((ptr) + ((ptr) - (OpusEncoder **)(ptr)))
#define OPUS_MULTISTREAM_GET_ENCODER_STATE(x, y) OPUS_MULTISTREAM_GET_ENCODER_STATE_REQUEST, __opus_check_int(x), __opus_check_encstate_ptr(y)
/* The size of this library's block: a header and `streams` OpusEncoder blocks (not libopus's size). */
opus_int32 opus_multistream_encoder_get_size(int streams, int coupled_streams);
opus_int32 opus_multistream_surround_encoder_get_size(int channels, int mapping_family);
OpusMSEncoder *opus_multistream_encoder_create(opus_int32 Fs, int channels, int streams, int coupled_streams, const unsigned char *mapping,
                                               int application, int *error);
OpusMSEncoder *opus_multistream_surround_encoder_create(opus_int32 Fs, int channels, int mapping_family, int *streams, int *coupled_streams,
                                                        unsigned char *mapping, int application, int *error);
int opus_multistream_encoder_init(OpusMSEncoder *st, opus_int32 Fs, int channels, int streams, int coupled_streams, const unsigned char *mapping,
                                  int application);
int opus_multistream_surround_encoder_init(OpusMSEncoder *st, opus_int32 Fs, int channels, int mapping_family, int *streams, int *coupled_streams,
                                           unsigned char *mapping, int application);
/* Returns the packet length or an error: OPUS_BAD_ARG for a frame size no stream codes, OPUS_BUFFER_TOO_SMALL when
 * max_data_bytes < 4*streams - 1. */
opus_int32 opus_multistream_encode(OpusMSEncoder *st, const opus_int16 *pcm, int frame_size, unsigned char *data, opus_int32 max_data_bytes);
/* OPUS_SET_BITRATE sets the multistream bitrate (OPUS_AUTO, OPUS_BITRATE_MAX or >= 0, not clamped); OPUS_GET_BITRATE is the sum of
 * the streams' bitrates and OPUS_GET_FINAL_RANGE the XOR of their final ranges; OPUS_RESET_STATE and the other SETs go to every
 * stream, the other GETs are answered by stream 0; OPUS_MULTISTREAM_GET_ENCODER_STATE(id, &enc) gives the embedded OpusEncoder of
 * stream id, on which opus_encoder_ctl works. */
int opus_multistream_encoder_ctl(OpusMSEncoder *st, int request, ...);
void opus_multistream_encoder_destroy(OpusMSEncoder *st);

/* Multistream encode spans (ours), the contracts of opus_encode_span / _span_device / opus_encoder_sync: PCM of frame (m,f) at
 * pcm + (m*F+f)*frame_size*channels, its packet at data + (m*F+f)*max_data_bytes, ret[m*F+f] what opus_multistream_encode returns.
 * Every encoder of a span shares Fs, channels, streams and coupled_streams; mappings and settings may differ.  _device: pcm / data /
 * ret are DEVICE pointers and the call only enqueues on the encoder stream (except in CBR, where it waits for the call to read the
 * last stream's final bitrate back); opus_b200_enc_synchronize() waits. */
int opus_multistream_encode_span(OpusMSEncoder **st, int n, int F, const opus_int16 *pcm, int frame_size, unsigned char *data,
                                 opus_int32 max_data_bytes, opus_int32 *ret);
int opus_multistream_encode_span_device(OpusMSEncoder **st, int n, int F, const opus_int16 *d_pcm, int frame_size, unsigned char *d_data,
                                        opus_int32 max_data_bytes, opus_int32 *d_ret);
int opus_multistream_encoder_sync(OpusMSEncoder **st, int n);

/* ---- runtime ---- */
int opus_b200_init(int device);            /* select the CUDA device (default 0); 0 or OPUS_INTERNAL_ERROR */
int opus_b200_synchronize(void);
void *opus_b200_stream(void);              /* the cudaStream_t the library launches on (for event timing) */
long long opus_b200_kernel_launches(void); /* number of codec kernels launched so far by this process */
/* Accumulated device time per pipeline stage (0 parse, 1 synth, 2 de-emphasis) in ms and launches, since the last reset. */
int opus_b200_stage_times(double ms[3], long long launches[3], int reset);
/* The same for the two stages of multistream calls (0 split, 1 gather). */
int opus_b200_ms_stage_times(double ms[2], long long launches[2], int reset);
/* The same for the multistream encoder's kernels (0 route, 1 budget, 2 pack), on the encoder stream. */
int opus_b200_ms_enc_stage_times(double ms[3], long long launches[3], int reset);
/* Time of the last span call in milliseconds, from CUDA events recorded around it on the library stream. */
float opus_b200_last_kernel_ms(void);
int opus_b200_device_index(void);         /* device in use, -1 when CUDA is unusable */
/* encoder half: its own stream */
int opus_b200_enc_synchronize(void);
void *opus_b200_enc_stream(void);          /* the cudaStream_t the encoder launches on */
long long opus_b200_enc_kernel_launches(void);
float opus_b200_enc_last_kernel_ms(void);  /* device time of the last encode span (CUDA events on the encoder stream) */
/* The encoder has two device paths: the frame-synchronous kernel pipeline (OPUS_APPLICATION_RESTRICTED_LOWDELAY streams, frames
 * up to 20 ms) and a one-kernel path for everything else; both are bit-exact with the reference.  set_pipeline(0) sends every
 * stream through the one-kernel path (A/B measurements, tests); returns the previous setting.  path_counts: streams x calls
 * each path has coded so far. */
int opus_b200_enc_set_pipeline(int on);
void opus_b200_enc_path_counts(long long *pipeline, long long *one_kernel);
/* The pipeline's band loop runs a budget-only chain first, searches every leaf it lists in parallel, then the exact chain;
 * a leaf whose pulse count the exact chain finds different is searched there.  Counters since start (synchronises). */
void opus_b200_enc_band_stats(long long *searched_by_exact_chain, long long *leaves_listed);

#ifdef __cplusplus
}
#endif
#endif /* OPUS_B200_H */

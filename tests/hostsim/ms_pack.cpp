// tests/hostsim/ms_pack.cpp — TEST TOOL, never part of the product library.
//
// The multistream encoder's host-and-device functions (concentus_b200/csrc/opus_ms_encoder.h, and ms_pack_packet of
// opus_multistream.h, what ms_pack_kernel runs per stream of a packet) compiled for the CPU, so that `pytest -m "not gpu"` checks
// the layout rules, the rate allocation, the byte budgets and the framing.
#include "../../concentus_b200/csrc/celt_simt.cuh"   // CB_NOUNROLL for opus_packet.h, as csrc/opus_repacketizer.cu includes it
#include "../../concentus_b200/csrc/opus_ms_encoder.h"
#include "../../concentus_b200/csrc/opus_multistream.h"

extern "C" {

int hostsim_ms_pack(const uint8_t *pkt, int32_t len, int self_delimited, int pad, uint8_t *out, int32_t maxlen) {
    return cb::ms_pack_packet(pkt, len, self_delimited, pad, out, maxlen);
}
int hostsim_ms_check_layout(int channels, int streams, int coupled, const uint8_t *mapping) {
    return cb::ms_enc_check_layout(channels, streams, coupled, mapping);
}
int hostsim_ms_surround_layout(int channels, int family, int *streams, int *coupled, uint8_t *mapping) {
    return cb::ms_surround_layout(channels, family, streams, coupled, mapping);
}
void hostsim_ms_rate_allocation(int B, int channels, int streams, int coupled, int Fs, int frame_size, int32_t *rate) {
    cb::ms_rate_allocation(B, channels, streams, coupled, Fs, frame_size, rate);
}
int hostsim_ms_cbr_max_bytes(int max_data_bytes, int B, int Fs, int frame_size) { return cb::ms_cbr_max_bytes(max_data_bytes, B, Fs, frame_size); }
int hostsim_ms_stream_budget(int max_data_bytes, int tot_size, int streams, int s) { return cb::ms_stream_budget(max_data_bytes, tot_size, streams, s); }
int hostsim_ms_cbr_last_bitrate(int curr_max, int Fs, int frame_size) { return cb::ms_cbr_last_bitrate(curr_max, Fs, frame_size); }
int hostsim_ms_min_bytes(int streams) { return cb::ms_enc_min_bytes(streams); }
}

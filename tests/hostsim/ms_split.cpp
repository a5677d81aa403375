// tests/hostsim/ms_split.cpp — TEST TOOL, never part of the product library.
//
// The multistream packet split of concentus_b200/csrc/opus_multistream.h (what ms_split_kernel runs per packet) compiled for the
// CPU, so that `pytest -m "not gpu"` checks its validation codes and the undelimited packets it writes.
#include <cstring>
#include "../../concentus_b200/csrc/celt_simt.cuh"   // CB_NOUNROLL for opus_packet.h, as csrc/opus_repacketizer.cu includes it
#include "../../concentus_b200/csrc/opus_multistream.h"

extern "C" {

// `out` (len + 2 bytes at least) receives a copy of the packet with the sub-packets of streams 0..S-2 rewritten undelimited, and
// the reject marker after it; stream s's packet is out[eoffs[s]..][0..elens[s]).  Returns what ms_split_packet returns.
int hostsim_ms_split(const uint8_t *data, int32_t len, int S, int Fs, int frame_size, uint8_t *out, int64_t *eoffs, int32_t *elens) {
    const int64_t n = len > 0 ? len : 0;
    if (n > 0) memcpy(out, data, (size_t)n);
    cb::ms_write_reject_marker(out + n);
    return cb::ms_split_packet(data, len, S, Fs, frame_size, out, 0, eoffs, elens, 1, n);
}
}

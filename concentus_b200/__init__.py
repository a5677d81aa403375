"""concentus_b200 — B200-native batched CELT (Opus) codec engine.

The product is libconcentus_b200.so (hand-written sm_100a CUDA + a libopus-compatible C ABI, see
include/opus_b200.h).  This package is only the thin Python binding used by the tests and bench.py: it
loads the shared library with ctypes and mirrors the C entry points one-to-one.  It never falls back
to a CPU implementation: if the library is missing it raises, and on a box without a usable CUDA device
every codec call returns OPUS_INTERNAL_ERROR.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CB200_LIB", os.path.join(HERE, "libconcentus_b200.so"))   # override: A/B builds only

OPUS_OK = 0
OPUS_BAD_ARG = -1
OPUS_BUFFER_TOO_SMALL = -2
OPUS_INTERNAL_ERROR = -3
OPUS_INVALID_PACKET = -4
OPUS_UNIMPLEMENTED = -5
OPUS_INVALID_STATE = -6
OPUS_ALLOC_FAIL = -7
OPUS_RESET_STATE = 4028
OPUS_GET_FINAL_RANGE_REQUEST = 4031
OPUS_GET_BANDWIDTH_REQUEST = 4009
OPUS_GET_SAMPLE_RATE_REQUEST = 4029
OPUS_GET_PITCH_REQUEST = 4033
OPUS_SET_GAIN_REQUEST = 4034
OPUS_GET_GAIN_REQUEST = 4045
OPUS_GET_LAST_PACKET_DURATION_REQUEST = 4039
OPUS_MULTISTREAM_GET_DECODER_STATE_REQUEST = 5122
OPUS_MULTISTREAM_GET_ENCODER_STATE_REQUEST = 5120
OPUS_GET_BITRATE_REQUEST = 4003

_lib = None

EXPORTS = [
    "opus_decoder_get_size", "opus_decoder_create", "opus_decoder_init", "opus_decode", "opus_decoder_ctl",
    "opus_decoder_destroy", "opus_packet_parse", "opus_packet_get_bandwidth", "opus_packet_get_samples_per_frame",
    "opus_packet_get_nb_channels", "opus_packet_get_nb_frames", "opus_packet_get_nb_samples",
    "opus_decoder_get_nb_samples", "opus_strerror", "opus_get_version_string", "opus_decode_batch", "opus_decode_span",
    "opus_decode_span_device", "opus_decoder_sync", "opus_b200_init", "opus_b200_synchronize", "opus_b200_stream",
    "opus_b200_kernel_launches", "opus_b200_last_kernel_ms", "opus_b200_stage_times", "opus_b200_device_index",
    "opus_encoder_get_size", "opus_encoder_create", "opus_encoder_init", "opus_encode", "opus_encoder_ctl", "opus_encoder_destroy",
    "opus_packet_pad", "opus_packet_unpad", "opus_encode_batch", "opus_encode_span", "opus_encode_span_device", "opus_encode_span_ranges", "opus_encoder_sync",
    "opus_b200_enc_synchronize", "opus_b200_enc_stream", "opus_b200_enc_kernel_launches", "opus_b200_enc_last_kernel_ms",
    "opus_repacketizer_get_size", "opus_repacketizer_init", "opus_repacketizer_create", "opus_repacketizer_destroy", "opus_repacketizer_cat",
    "opus_repacketizer_get_nb_frames", "opus_repacketizer_out_range", "opus_repacketizer_out",
    "opus_b200_enc_set_pipeline", "opus_b200_enc_path_counts", "opus_b200_enc_band_stats",
    "opus_multistream_decoder_get_size", "opus_multistream_decoder_create", "opus_multistream_decoder_init", "opus_multistream_decode",
    "opus_multistream_decoder_ctl", "opus_multistream_decoder_destroy", "opus_multistream_decode_span",
    "opus_multistream_decode_span_device", "opus_multistream_decoder_sync", "opus_b200_ms_stage_times",
    "opus_multistream_encoder_get_size", "opus_multistream_encoder_create", "opus_multistream_encoder_init", "opus_multistream_encode",
    "opus_multistream_encoder_ctl", "opus_multistream_encoder_destroy", "opus_multistream_surround_encoder_get_size",
    "opus_multistream_surround_encoder_create", "opus_multistream_surround_encoder_init", "opus_multistream_encode_span",
    "opus_multistream_encode_span_device", "opus_multistream_encoder_sync", "opus_b200_ms_enc_stage_times",
]

OPUS_APPLICATION_VOIP = 2048
OPUS_APPLICATION_AUDIO = 2049
OPUS_APPLICATION_RESTRICTED_LOWDELAY = 2051
OPUS_AUTO = -1000
OPUS_SET_BITRATE_REQUEST = 4002
OPUS_SET_VBR_REQUEST = 4006
OPUS_SET_BANDWIDTH_REQUEST = 4008
OPUS_SET_COMPLEXITY_REQUEST = 4010
OPUS_SET_VBR_CONSTRAINT_REQUEST = 4020
OPUS_SET_FORCE_CHANNELS_REQUEST = 4022
OPUS_SET_FORCE_MODE_REQUEST = 11002


def lib():
    """Load the CUDA library (building is __graft_entry__.build()'s job).  Raises if it is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError("libconcentus_b200.so is not built (run `python -m concentus_b200.build`); "
                               "there is no CPU fallback")
        L = C.CDLL(LIB_PATH)
        L.opus_decoder_create.restype = C.c_void_p
        L.opus_decoder_create.argtypes = [C.c_int32, C.c_int, C.POINTER(C.c_int)]
        L.opus_decoder_init.argtypes = [C.c_void_p, C.c_int32, C.c_int]
        L.opus_decoder_destroy.argtypes = [C.c_void_p]
        L.opus_decoder_destroy.restype = None
        L.opus_decode.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_int, C.c_int]
        L.opus_decode_span.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_int, C.c_void_p]
        L.opus_decode_span_device.argtypes = L.opus_decode_span.argtypes
        L.opus_decode_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int]
        L.opus_decoder_sync.argtypes = [C.c_void_p, C.c_int]
        L.opus_strerror.restype = C.c_char_p
        L.opus_get_version_string.restype = C.c_char_p
        L.opus_b200_stream.restype = C.c_void_p
        L.opus_b200_kernel_launches.restype = C.c_longlong
        L.opus_b200_last_kernel_ms.restype = C.c_float
        L.opus_b200_stage_times.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        L.opus_encoder_create.restype = C.c_void_p
        L.opus_encoder_create.argtypes = [C.c_int32, C.c_int, C.c_int, C.POINTER(C.c_int)]
        L.opus_encoder_init.argtypes = [C.c_void_p, C.c_int32, C.c_int, C.c_int]
        L.opus_encoder_destroy.argtypes = [C.c_void_p]
        L.opus_encoder_destroy.restype = None
        L.opus_encode.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int32]
        L.opus_encode_span.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int32, C.c_void_p]
        L.opus_encode_span_device.argtypes = L.opus_encode_span.argtypes
        L.opus_encode_span_ranges.argtypes = L.opus_encode_span.argtypes + [C.c_void_p]
        L.opus_encode_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int32, C.c_void_p, C.c_int]
        L.opus_encoder_sync.argtypes = [C.c_void_p, C.c_int]
        L.opus_packet_pad.argtypes = [C.c_void_p, C.c_int32, C.c_int32]
        L.opus_packet_unpad.argtypes = [C.c_void_p, C.c_int32]
        L.opus_b200_enc_kernel_launches.restype = C.c_longlong
        L.opus_b200_enc_stream.restype = C.c_void_p
        L.opus_b200_enc_last_kernel_ms.restype = C.c_float
        L.opus_multistream_decoder_create.restype = C.c_void_p
        L.opus_multistream_decoder_create.argtypes = [C.c_int32, C.c_int, C.c_int, C.c_int, C.c_void_p, C.POINTER(C.c_int)]
        L.opus_multistream_decoder_init.argtypes = [C.c_void_p, C.c_int32, C.c_int, C.c_int, C.c_int, C.c_void_p]
        L.opus_multistream_decoder_get_size.argtypes = [C.c_int, C.c_int]
        L.opus_multistream_decoder_destroy.argtypes = [C.c_void_p]
        L.opus_multistream_decoder_destroy.restype = None
        L.opus_multistream_decode.argtypes = L.opus_decode.argtypes
        L.opus_multistream_decode_span.argtypes = L.opus_decode_span.argtypes
        L.opus_multistream_decode_span_device.argtypes = L.opus_decode_span.argtypes
        L.opus_multistream_decoder_sync.argtypes = [C.c_void_p, C.c_int]
        L.opus_b200_ms_stage_times.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        L.opus_multistream_encoder_create.restype = C.c_void_p
        L.opus_multistream_encoder_create.argtypes = [C.c_int32, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.POINTER(C.c_int)]
        L.opus_multistream_encoder_init.argtypes = [C.c_void_p, C.c_int32, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int]
        L.opus_multistream_encoder_get_size.argtypes = [C.c_int, C.c_int]
        L.opus_multistream_surround_encoder_get_size.argtypes = [C.c_int, C.c_int]
        L.opus_multistream_surround_encoder_create.restype = C.c_void_p
        L.opus_multistream_surround_encoder_create.argtypes = [C.c_int32, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                                               C.POINTER(C.c_int)]
        L.opus_multistream_surround_encoder_init.argtypes = [C.c_void_p, C.c_int32, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                                             C.c_int]
        L.opus_multistream_encoder_destroy.argtypes = [C.c_void_p]
        L.opus_multistream_encoder_destroy.restype = None
        L.opus_multistream_encode.argtypes = L.opus_encode.argtypes
        L.opus_multistream_encode_span.argtypes = L.opus_encode_span.argtypes
        L.opus_multistream_encode_span_device.argtypes = L.opus_encode_span.argtypes
        L.opus_multistream_encoder_sync.argtypes = [C.c_void_p, C.c_int]
        L.opus_b200_ms_enc_stage_times.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        _lib = L
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


class DecoderBatch:
    """n independent decoders (same Fs / channels) driven through the batch C ABI."""

    def __init__(self, n, Fs=48000, channels=2):
        L = lib()
        self.n, self.Fs, self.channels = n, Fs, channels
        err = C.c_int(0)
        self.handles = (C.c_void_p * n)()
        for i in range(n):
            h = L.opus_decoder_create(Fs, channels, C.byref(err))
            if not h:
                raise RuntimeError("opus_decoder_create failed: %d" % err.value)
            self.handles[i] = h

    def decode_span(self, data, offs, lens, F, frame_size):
        """Host buffers in, host buffers out: returns (pcm [n*F*frame_size, channels], rets [n*F])."""
        L = lib()
        pcm = np.zeros((self.n * F * frame_size, self.channels), dtype=np.int16)
        rets = np.zeros(self.n * F, dtype=np.int32)
        rc = L.opus_decode_span(self.handles, self.n, F, _p(data), _p(np.ascontiguousarray(offs, dtype=np.int64)),
                                _p(np.ascontiguousarray(lens, dtype=np.int32)), _p(pcm), frame_size, _p(rets))
        if rc != OPUS_OK:
            raise RuntimeError("opus_decode_span: %s" % L.opus_strerror(rc).decode())
        return pcm, rets

    def final_ranges(self):
        L = lib()
        out = np.zeros(self.n, dtype=np.uint32)
        v = C.c_uint32(0)
        for i in range(self.n):
            L.opus_decoder_ctl(C.c_void_p(self.handles[i]), OPUS_GET_FINAL_RANGE_REQUEST, C.byref(v))
            out[i] = v.value
        return out

    def close(self):
        L = lib()
        for i in range(self.n):
            if self.handles[i]:
                L.opus_decoder_destroy(C.c_void_p(self.handles[i]))
                self.handles[i] = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class MSDecoderBatch:
    """n multistream decoders (same Fs / channels / streams / coupled streams) driven through the multistream span C ABI.
    mapping: one channel mapping for all decoders, or one per decoder."""

    def __init__(self, n, Fs, channels, streams, coupled, mapping):
        L = lib()
        self.n, self.Fs, self.channels, self.streams, self.coupled = n, Fs, channels, streams, coupled
        maps = np.asarray(mapping, dtype=np.uint8).reshape(-1, channels)
        if maps.shape[0] == 1:
            maps = np.repeat(maps, n, axis=0)
        assert maps.shape[0] == n
        self.mappings = np.ascontiguousarray(maps)
        err = C.c_int(0)
        self.handles = (C.c_void_p * n)()
        for i in range(n):
            h = L.opus_multistream_decoder_create(Fs, channels, streams, coupled, _p(self.mappings[i]), C.byref(err))
            if not h:
                raise RuntimeError("opus_multistream_decoder_create failed: %d" % err.value)
            self.handles[i] = h

    def decode_span(self, data, offs, lens, F, frame_size):
        """Host buffers in, host buffers out: returns (pcm [n*F*frame_size, channels], rets [n*F])."""
        L = lib()
        pcm = np.zeros((self.n * F * frame_size, self.channels), dtype=np.int16)
        rets = np.zeros(self.n * F, dtype=np.int32)
        rc = L.opus_multistream_decode_span(self.handles, self.n, F, _p(data), _p(np.ascontiguousarray(offs, dtype=np.int64)),
                                            _p(np.ascontiguousarray(lens, dtype=np.int32)), _p(pcm), frame_size, _p(rets))
        if rc != OPUS_OK:
            raise RuntimeError("opus_multistream_decode_span: %s" % L.opus_strerror(rc).decode())
        return pcm, rets

    def final_ranges(self):
        """OPUS_GET_FINAL_RANGE of each multistream decoder: the XOR of its streams' final ranges."""
        L = lib()
        out = np.zeros(self.n, dtype=np.uint32)
        v = C.c_uint32(0)
        for i in range(self.n):
            L.opus_multistream_decoder_ctl(C.c_void_p(self.handles[i]), OPUS_GET_FINAL_RANGE_REQUEST, C.byref(v))
            out[i] = v.value
        return out

    def close(self):
        L = lib()
        for i in range(self.n):
            if self.handles[i]:
                L.opus_multistream_decoder_destroy(C.c_void_p(self.handles[i]))
                self.handles[i] = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class MSEncoderBatch:
    """n multistream encoders (same Fs / channels / streams / coupled streams) driven through the multistream span C ABI.
    mapping: one channel mapping for all encoders, or one per encoder.  bitrate is the multistream bitrate; vbr / cvbr /
    complexity go to every stream."""

    def __init__(self, n, Fs, channels, streams, coupled, mapping, application=OPUS_APPLICATION_RESTRICTED_LOWDELAY, bitrate=OPUS_AUTO,
                 vbr=1, cvbr=1, complexity=9):
        L = lib()
        self.n, self.Fs, self.channels, self.streams, self.coupled = n, Fs, channels, streams, coupled
        maps = np.asarray(mapping, dtype=np.uint8).reshape(-1, channels)
        if maps.shape[0] == 1:
            maps = np.repeat(maps, n, axis=0)
        assert maps.shape[0] == n
        self.mappings = np.ascontiguousarray(maps)
        err = C.c_int(0)
        self.handles = (C.c_void_p * n)()
        for i in range(n):
            h = L.opus_multistream_encoder_create(Fs, channels, streams, coupled, _p(self.mappings[i]), application, C.byref(err))
            if not h:
                raise RuntimeError("opus_multistream_encoder_create failed: %d" % err.value)
            self.handles[i] = h
            for req, v in ((OPUS_SET_BITRATE_REQUEST, bitrate), (OPUS_SET_VBR_REQUEST, vbr), (OPUS_SET_VBR_CONSTRAINT_REQUEST, cvbr),
                           (OPUS_SET_COMPLEXITY_REQUEST, complexity)):
                rc = L.opus_multistream_encoder_ctl(C.c_void_p(h), req, C.c_int32(v))
                if rc != OPUS_OK:
                    raise RuntimeError("opus_multistream_encoder_ctl(%d, %d) -> %d" % (req, v, rc))

    def encode_span(self, pcm, F, frame_size, max_data_bytes):
        """pcm: int16 [n*F*frame_size, channels] (encoder-major).  Returns (data uint8 [n*F, max_data_bytes], rets int32 [n*F])."""
        L = lib()
        pcm = np.ascontiguousarray(pcm, dtype=np.int16)
        assert pcm.size == self.n * F * frame_size * self.channels
        data = np.zeros((self.n * F, max_data_bytes), dtype=np.uint8)
        rets = np.zeros(self.n * F, dtype=np.int32)
        rc = L.opus_multistream_encode_span(self.handles, self.n, F, _p(pcm), frame_size, _p(data), max_data_bytes, _p(rets))
        if rc != OPUS_OK:
            raise RuntimeError("opus_multistream_encode_span: %s" % L.opus_strerror(rc).decode())
        return data, rets

    def _get(self, request):
        L = lib()
        out = np.zeros(self.n, dtype=np.uint32 if request == OPUS_GET_FINAL_RANGE_REQUEST else np.int32)
        v = C.c_int32(0)
        for i in range(self.n):
            rc = L.opus_multistream_encoder_ctl(C.c_void_p(self.handles[i]), request, C.byref(v))
            if rc != OPUS_OK:
                raise RuntimeError("opus_multistream_encoder_ctl(%d) -> %d" % (request, rc))
            out[i] = v.value & 0xFFFFFFFF if request == OPUS_GET_FINAL_RANGE_REQUEST else v.value
        return out

    def final_ranges(self):
        """OPUS_GET_FINAL_RANGE of each multistream encoder: the XOR of its streams' final ranges."""
        return self._get(OPUS_GET_FINAL_RANGE_REQUEST)

    def bitrates(self):
        """OPUS_GET_BITRATE of each multistream encoder: the sum of its streams' bitrates."""
        return self._get(OPUS_GET_BITRATE_REQUEST)

    def close(self):
        L = lib()
        for i in range(self.n):
            if self.handles[i]:
                L.opus_multistream_encoder_destroy(C.c_void_p(self.handles[i]))
                self.handles[i] = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class EncoderBatch:
    """n independent encoders (same Fs / channels / settings) driven through the batch C ABI."""

    def __init__(self, n, Fs=48000, channels=2, application=OPUS_APPLICATION_RESTRICTED_LOWDELAY, bitrate=OPUS_AUTO, vbr=1, cvbr=1,
                 complexity=9, force_channels=0, bandwidth=0, force_mode=0):
        L = lib()
        self.n, self.Fs, self.channels = n, Fs, channels
        err = C.c_int(0)
        self.handles = (C.c_void_p * n)()
        for i in range(n):
            h = L.opus_encoder_create(Fs, channels, application, C.byref(err))
            if not h:
                raise RuntimeError("opus_encoder_create failed: %d" % err.value)
            self.handles[i] = h
            hp = C.c_void_p(h)
            for req, v in ((OPUS_SET_BITRATE_REQUEST, bitrate), (OPUS_SET_VBR_REQUEST, vbr), (OPUS_SET_VBR_CONSTRAINT_REQUEST, cvbr),
                           (OPUS_SET_COMPLEXITY_REQUEST, complexity)):
                rc = L.opus_encoder_ctl(hp, req, C.c_int32(v))
                if rc != OPUS_OK:
                    raise RuntimeError("opus_encoder_ctl(%d, %d) -> %d" % (req, v, rc))
            if force_channels:
                L.opus_encoder_ctl(hp, OPUS_SET_FORCE_CHANNELS_REQUEST, C.c_int32(force_channels))
            if bandwidth:
                L.opus_encoder_ctl(hp, OPUS_SET_BANDWIDTH_REQUEST, C.c_int32(bandwidth))
            if force_mode:
                L.opus_encoder_ctl(hp, OPUS_SET_FORCE_MODE_REQUEST, C.c_int32(force_mode))

    def encode_span(self, pcm, F, frame_size, max_data_bytes=1276):
        """pcm: int16 [n*F*frame_size, channels] (stream-major).  Returns (data uint8 [n*F, max_data_bytes], lens int32 [n*F])."""
        L = lib()
        pcm = np.ascontiguousarray(pcm, dtype=np.int16)
        assert pcm.size == self.n * F * frame_size * self.channels
        data = np.zeros((self.n * F, max_data_bytes), dtype=np.uint8)
        lens = np.zeros(self.n * F, dtype=np.int32)
        rc = L.opus_encode_span(self.handles, self.n, F, _p(pcm), frame_size, _p(data), max_data_bytes, _p(lens))
        if rc != OPUS_OK:
            raise RuntimeError("opus_encode_span: %s" % L.opus_strerror(rc).decode())
        return data, lens

    def final_ranges(self):
        L = lib()
        out = np.zeros(self.n, dtype=np.uint32)
        v = C.c_uint32(0)
        for i in range(self.n):
            L.opus_encoder_ctl(C.c_void_p(self.handles[i]), OPUS_GET_FINAL_RANGE_REQUEST, C.byref(v))
            out[i] = v.value
        return out

    def close(self):
        L = lib()
        for i in range(self.n):
            if self.handles[i]:
                L.opus_encoder_destroy(C.c_void_p(self.handles[i]))
                self.handles[i] = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

// tests/hostsim/hostsim.cpp — TEST TOOL, never part of the product library.
//
// Compiles the codec headers of concentus_b200/csrc with a plain C++ compiler (1-lane teams, see
// celt_simt.cuh) so the integer semantics of both pipeline stages can be diffed against the oracle on a
// machine with no GPU.  The CUDA build of the very same headers is what ships; this file exists
// only so `pytest -m "not gpu"` can localise a bit mismatch before GPU time is spent.
#include <cstdlib>
#include <cstring>
#include <vector>
#include "../../concentus_b200/csrc/opus_decoder_dev.cuh"

extern "C" {

// The tests' music signal (tests/oracle_lib.py generate_music), the same function as ref_generate_music in oracle/ref_harness.c:
// opus-fix/tests/test_opus_encode.c:59-90 driven by the MWC generator of tests/test_opus_common.h:55-62 with an explicit seed.
void hostsim_generate_music(int16_t *buf, int32_t len, uint32_t seed) {
    uint32_t Rz = seed, Rw = seed;
    int32_t a1 = 0, b1 = 0, a2 = 0, b2 = 0, c1 = 0, c2 = 0, d1 = 0, d2 = 0, j = 0;
    for (int32_t i = 0; i < len; i++) {
        uint32_t r;
        int32_t v1, v2;
        v1 = v2 = (((j * ((j >> 12) ^ ((j >> 10 | j >> 12) & 26 & j >> 7))) & 128) + 128) << 15;
        Rz = 36969 * (Rz & 65535) + (Rz >> 16); Rw = 18000 * (Rw & 65535) + (Rw >> 16);
        r = (Rz << 16) + Rw; v1 += r & 65535; v1 -= r >> 16;
        Rz = 36969 * (Rz & 65535) + (Rz >> 16); Rw = 18000 * (Rw & 65535) + (Rw >> 16);
        r = (Rz << 16) + Rw; v2 += r & 65535; v2 -= r >> 16;
        b1 = v1 - a1 + ((b1 * 61 + 32) >> 6); a1 = v1;
        b2 = v2 - a2 + ((b2 * 61 + 32) >> 6); a2 = v2;
        c1 = (30 * (c1 + b1 + d1) + 32) >> 6; d1 = b1;
        c2 = (30 * (c2 + b2 + d2) + 32) >> 6; d2 = b2;
        v1 = (c1 + 128) >> 8;
        v2 = (c2 + 128) >> 8;
        buf[i * 2] = v1 > 32767 ? 32767 : (v1 < -32768 ? -32768 : v1);
        buf[i * 2 + 1] = v2 > 32767 ? 32767 : (v2 < -32768 ? -32768 : v2);
        if (i % 6 == 0) j++;
    }
}

int hostsim_dec_state_size(void) { return (int)sizeof(CbDecState); }

// Decode F packets of one stream (packed layout).  cap = pcm capacity per packet (samples per channel).
// Stage A (parse -> IR), stage B (synth) and stage C (de-emphasis) per packet, exactly the hand-offs the kernels use.
// bounds (nb entries, ascending, last = F) are the ends of the emulated calls; nullptr = calls of 16 packets.
int hostsim_decode_stream_calls(const uint8_t *data, const int64_t *offs, const int32_t *lens, int F, int cap, int channels,
                                int Fs, int16_t *pcm, uint32_t *ranges, int32_t *rets, const int *bounds, int nb) {
    // Emulates the kernels' schedule: the call is cut into chunks of Fc packets; for a chunk, stage A runs first for every run
    // of R packets from the state as it stood when the chunk began (each run reconstructing its own context), then stages B
    // and C consume the chunk in order.  (The kernels use the state at CALL start for all chunks and walk back across chunk
    // boundaries inside the call; a chunk here is therefore a "call".)
    const int Fc = 16, R = 3;
    CbDecState *st = (CbDecState *)calloc(1, sizeof(CbDecState));
    cb::SynthScratch *S = (cb::SynthScratch *)calloc(1, sizeof(cb::SynthScratch));
    cb::ParseScratch *ps = (cb::ParseScratch *)calloc(1, sizeof(cb::ParseScratch));
    cb::PlcScratch *plc = (cb::PlcScratch *)calloc(1, sizeof(cb::PlcScratch));
    if (cb::dec_state_init(st, Fs, channels) != 0) return -1;
    const int kmax = cap / (Fs / 400) < 48 ? (cap / (Fs / 400) > 0 ? cap / (Fs / 400) : 1) : 48;
    const int xstride = cap * (48000 / Fs) * 2 + 16;
    std::vector<CbPacketIR> pk(Fc);
    std::vector<CbFrameIR> fr((size_t)Fc * kmax);
    std::vector<int16_t> X((size_t)Fc * xstride);
    std::vector<int> sig((size_t)cap * (48000 / Fs) * 2 + 16);
    cb::SoloTeam tm;
    int bi = 0;
    for (int f0 = 0; f0 < F;) {
        int f1 = f0 + Fc < F ? f0 + Fc : F;
        if (bounds) f1 = bi < nb ? bounds[bi++] : F;
        if ((size_t)(f1 - f0) > pk.size()) {
            pk.resize(f1 - f0);
            fr.resize((size_t)(f1 - f0) * kmax);
            X.resize((size_t)(f1 - f0) * xstride);
        }
        cb::CbCallCtx c0;
        cb::call_ctx_from_state(c0, st);
        for (int first = f0; first < f1; first += R)   // stage A, run by run, any order
            cb::opus_parse_run(c0, data, offs, lens, f0, first, first + R < f1 ? first + R : f1, cap, 0, kmax, xstride, pk.data(), fr.data(),
                               X.data(), f0, *ps);
        for (int f = f0; f < f1; f++) {                // stages B and C
            const int slot = f - f0;
            cb::CbSigRange rg;
            int r = cb::opus_synth_packet(tm, st, *S, *plc, pk[slot], fr.data() + (size_t)slot * kmax, X.data() + (size_t)slot * xstride,
                                          pcm + (size_t)f * cap * channels, cap, sig.data(), &rg);
            for (int c = 0; c < channels; c++) cb::opus_deemph_packet(st, c, sig.data(), rg, pcm + (size_t)f * cap * channels, cap);
            if (rets) rets[f] = r;
            if (ranges) ranges[f] = st->rangeFinal;
        }
        f0 = f1;
    }
    free(plc);
    free(ps);
    free(S);
    free(st);
    return 0;
}
int hostsim_decode_stream(const uint8_t *data, const int64_t *offs, const int32_t *lens, int F, int cap, int channels,
                          int Fs, int16_t *pcm, uint32_t *ranges, int32_t *rets) {
    return hostsim_decode_stream_calls(data, offs, lens, F, cap, channels, Fs, pcm, ranges, rets, nullptr, 0);
}
}

// ---- encoder ----------------------------------------------------------------------------------------------------
#include "../../concentus_b200/csrc/opus_encoder_dev.cuh"

extern "C" {

int hostsim_enc_state_size(void) { return (int)sizeof(CbEncState); }

// Encode F frames of one stream with the 1-lane team.  cfg = {application, bitrate, vbr, cvbr, complexity, max_bytes,
// force_channels, bandwidth} (the oracle harness's ref_enc_cfg).  out: F slots of `stride` bytes.
int hostsim_encode_stream(const int16_t *pcm, int F, int frame_size, int channels, int Fs, const int *cfg, uint8_t *out, int stride,
                          int32_t *lens, uint32_t *ranges) {
    CbEncState *st = (CbEncState *)calloc(1, sizeof(CbEncState));
    cb::EncShared *S = (cb::EncShared *)calloc(1, sizeof(cb::EncShared));
    cb::EncGlobal *G = (cb::EncGlobal *)calloc(1, sizeof(cb::EncGlobal));
    if (cb::enc_state_init(st, Fs, channels, cfg[0]) != 0) return -1;
    int dummy = 0;
    cb::enc_ctl(st, 4002, cfg[1], &dummy);
    cb::enc_ctl(st, 4006, cfg[2], &dummy);
    cb::enc_ctl(st, 4020, cfg[3], &dummy);
    cb::enc_ctl(st, 4010, cfg[4], &dummy);
    if (cfg[6]) cb::enc_ctl(st, 4022, cfg[6], &dummy);
    if (cfg[7]) cb::enc_ctl(st, 4008, cfg[7], &dummy);
    cb::SoloTeam tm;
    int rc = 0;
    for (int f = 0; f < F; f++) {
        int n = cb::opus_encode_frame(tm, st, st, *S, *G, pcm + (size_t)f * frame_size * channels, frame_size, out + (size_t)f * stride,
                                      cfg[5] < stride ? cfg[5] : stride);
        lens[f] = n;
        if (n < 0) { rc = n; break; }
        if (ranges) ranges[f] = st->rangeFinal;
    }
    free(G);
    free(S);
    free(st);
    return rc;
}
// Same with a ctl script (see oracle/ref_harness.c ref_encode_stream_script): K (request, value) pairs before every frame.
int hostsim_encode_stream_script(const int16_t *pcm, int F, int frame_size, int channels, int Fs, const int *cfg, const int32_t *script, int K,
                                 uint8_t *out, int stride, int32_t *lens, uint32_t *ranges) {
    CbEncState *st = (CbEncState *)calloc(1, sizeof(CbEncState));
    cb::EncShared *S = (cb::EncShared *)calloc(1, sizeof(cb::EncShared));
    cb::EncGlobal *G = (cb::EncGlobal *)calloc(1, sizeof(cb::EncGlobal));
    if (cb::enc_state_init(st, Fs, channels, cfg[0]) != 0) return -1;
    int dummy = 0;
    cb::enc_ctl(st, 4002, cfg[1], &dummy);
    cb::enc_ctl(st, 4006, cfg[2], &dummy);
    cb::enc_ctl(st, 4020, cfg[3], &dummy);
    cb::enc_ctl(st, 4010, cfg[4], &dummy);
    cb::SoloTeam tm;
    for (int f = 0; f < F; f++) {
        for (int k = 0; k < K; k++) {
            const int req = script[(f * K + k) * 2], val = script[(f * K + k) * 2 + 1];
            if (req != 0) cb::enc_ctl(st, req, val, &dummy);
        }
        lens[f] = cb::opus_encode_frame(tm, st, st, *S, *G, pcm + (size_t)f * frame_size * channels, frame_size, out + (size_t)f * stride,
                                        cfg[5] < stride ? cfg[5] : stride);
        if (ranges) ranges[f] = st->rangeFinal;
    }
    free(G);
    free(S);
    free(st);
    return 0;
}
}

// ---- encoder, frame-synchronous pipeline (celt_enc_pipe.cuh): the same slices the pipeline kernels run, 1-lane teams ----------
#include "../../concentus_b200/csrc/celt_enc_pipe.cuh"

static int g_band_mode = 1;          // 0: the band loop as one stage (pipe_bands); 1: prep / chain-S / leaves / chain-X; 2: prep + one inline walk
static long long g_leaves = 0, g_misses = 0, g_frames = 0;

extern "C" {

void hostsim_set_band_mode(int m) { g_band_mode = m; }
void hostsim_band_stats(long long *leaves, long long *misses, long long *frames, int reset) {
    if (leaves) *leaves = g_leaves;
    if (misses) *misses = g_misses;
    if (frames) *frames = g_frames;
    if (reset) g_leaves = g_misses = g_frames = 0;
}

// Encode F frames of one stream through the pipeline stages in chunks of Fc frames.  Returns -100 when the stream is not one
// the pipeline takes (the library then uses the one-kernel path), else 0.  Same cfg / outputs as hostsim_encode_stream.
int hostsim_encode_stream_pipe(const int16_t *pcm, int F, int frame_size, int channels, int Fs, const int *cfg, uint8_t *out, int stride,
                               int32_t *lens, uint32_t *ranges, int Fc) {
    CbEncState *st = (CbEncState *)calloc(1, sizeof(CbEncState));
    if (cb::enc_state_init(st, Fs, channels, cfg[0]) != 0) return -1;
    int dummy = 0;
    cb::enc_ctl(st, 4002, cfg[1], &dummy);
    cb::enc_ctl(st, 4006, cfg[2], &dummy);
    cb::enc_ctl(st, 4020, cfg[3], &dummy);
    cb::enc_ctl(st, 4010, cfg[4], &dummy);
    if (cfg[6]) cb::enc_ctl(st, 4022, cfg[6], &dummy);
    if (cfg[7]) cb::enc_ctl(st, 4008, cfg[7], &dummy);
    const int out_bytes = cfg[5] < stride ? cfg[5] : stride;
    if (!cb::enc_pipe_eligible(st, frame_size, out_bytes)) { free(st); return -100; }
    cb::PipeGeom g;
    g.n = 1; g.CC = channels; g.Fs = Fs; g.upsample = 48000 / Fs; g.fsz = frame_size; g.N = frame_size * g.upsample;
    for (g.LM = 0; g.LM <= 3; g.LM++) if ((120 << g.LM) == g.N) break;
    g.F = F; g.Fc = Fc; g.max_bytes = out_bytes < 1276 ? out_bytes : 1276; g.stride = stride;
    g.pstride = cb::kPipeHist + Fc * g.N;
    const int row = frame_size * channels;
    std::vector<int16_t> D((size_t)Fc * row);
    std::vector<int> P((size_t)channels * g.pstride);
    std::vector<cb::EncPlan> plans(Fc);
    std::vector<cb::FeFrame> fe(Fc);
    cb::EncPipeCtx *X = (cb::EncPipeCtx *)calloc(1, sizeof(cb::EncPipeCtx));
    cb::EncPipeBuf *B = (cb::EncPipeBuf *)calloc(1, sizeof(cb::EncPipeBuf));
    cb::PitchScratch *ps = (cb::PitchScratch *)calloc(1, sizeof(cb::PitchScratch));
    cb::TransformScratch *ts = (cb::TransformScratch *)calloc(1, sizeof(cb::TransformScratch));
    cb::BandScratch *bs = (cb::BandScratch *)calloc(1, sizeof(cb::BandScratch));
    cb::PrepScratch *prs = (cb::PrepScratch *)calloc(1, sizeof(cb::PrepScratch));
    cb::LeafScratch *lfs = (cb::LeafScratch *)calloc(1, sizeof(cb::LeafScratch));
    cb::BandPrep *bp = (cb::BandPrep *)calloc(1, sizeof(cb::BandPrep));
    cb::LeafList *ll = (cb::LeafList *)calloc(1, sizeof(cb::LeafList));
    cb::WalkScratch *ws = (cb::WalkScratch *)calloc(1, sizeof(cb::WalkScratch));
    std::vector<int16_t> xall(cb::kXallStride);
    std::vector<int> tin(960 + 120);
    int sc[4];
    cb::SoloTeam tm;
    for (int c = 0; c < channels; c++)
        for (int i = 0; i < cb::kPipeHist; i++) P[(size_t)c * g.pstride + i] = st->prefilter_mem[c * cb::kPipeHist + i];
    int rc = 0;
    for (int f0 = 0; f0 < F; f0 += Fc) {
        const int nfr = F - f0 < Fc ? F - f0 : Fc;
        // P0: the Opus layer of the chunk
        int m0[2] = {st->preemph_memE[0], st->preemph_memE[1]};
        for (int fi = 0; fi < nfr; fi++) {
            cb::pipe_plan_frame(st, pcm + (size_t)(f0 + fi) * row, frame_size, out_bytes, D.data() + (size_t)fi * row, plans[fi]);
            if (plans[fi].code)
                for (int c = 0; c < channels; c++) st->preemph_memE[c] = cb::pipe_preemph_mem_after(g, D.data() + (size_t)fi * row, c);
        }
        // FE1 / FE2, frame-parallel on the device
        for (int fi = 0; fi < nfr; fi++) {
            if (!plans[fi].code) continue;
            int mi[2];
            for (int c = 0; c < channels; c++) mi[c] = fi == 0 ? m0[c] : cb::pipe_preemph_mem_after(g, D.data() + (size_t)(fi - 1) * row, c);
            cb::pipe_preemph_frame(tm, g, plans[fi], D.data() + (size_t)fi * row, P.data(), fi, mi, fe[fi]);
        }
        for (int fi = nfr - 1; fi >= 0; fi--)   // any order
            cb::pipe_pitch_frame(tm, g, plans[fi], P.data() + fi * g.N, P.data() + g.pstride + fi * g.N, *ps, fe[fi]);
        // frame steps
        for (int fi = 0; fi < nfr; fi++) {
            uint8_t *o = out + (size_t)(f0 + fi) * stride;
            cb::pipe_head(st, g, plans[fi], fe[fi], *X, o);
            for (int c = 0; c < channels; c++) {
                int *inc = B->in + c * (g.N + cb::kOverlap);
                if ((f0 + fi) & 1) {
                    cb::pipe_comb_channel(tm, st, g, *X, P.data() + (size_t)c * g.pstride + fi * g.N, inc, c, tin.data(), sc);
                } else {   // the pipeline's form: comb only, then transient_analysis of the channel by one thread (odd / even frames alternate)
                    cb::pipe_comb_channel(tm, st, g, *X, P.data() + (size_t)c * g.pstride + fi * g.N, inc, c, nullptr, sc);
                    if (X->code && X->cfg.complexity >= 1) {
                        std::vector<int16_t> row(g.N + cb::kOverlap);
                        cb::TransientHp hp;
                        hp.reset();
                        for (int i = 0; i < g.N + cb::kOverlap; i++) row[i] = (int16_t)hp.step(inc[i] >> 12, i);
                        X->v.mask_metric[c] = cb::transient_finish_row(row.data(), g.N + cb::kOverlap, hp.mx, hp.mn);
                    }
                }
            }
            cb::pipe_transform(tm, st, g, *X, *B, *ts);
            cb::pipe_decide(st, g, *X);
            int r;
            if (g_band_mode == 0) {
                r = cb::pipe_bands(tm, st, g, plans[fi], *X, *B, *bs, o);
            } else if (g_band_mode == 2) {
                cb::pipe_band_prep(tm, st, g, *X, *B, *bp, xall.data(), *prs);
                r = cb::pipe_band_inline_finish(tm, st, g, plans[fi], *X, *bp, xall.data(), *ws, o);
            } else {
                cb::pipe_band_prep(tm, st, g, *X, *B, *bp, xall.data(), *prs);
                cb::pipe_band_spec(st, g, *X, *bp, *ll);
                cb::pipe_leaves(tm, st, *X, *ll, xall.data(), *lfs);
                int miss = 0;
                r = cb::pipe_band_exact_finish(st, g, plans[fi], *X, *bp, *ll, xall.data(), o, &miss);
                g_leaves += ll->count; g_misses += miss; g_frames++;
            }
            lens[f0 + fi] = r;
            if (r < 0) rc = r;
            if (ranges) ranges[f0 + fi] = st->rangeFinal;
        }
        // the chunk's tail of P is the next chunk's history
        for (int c = 0; c < channels; c++)
            for (int i = 0; i < cb::kPipeHist; i++) P[(size_t)c * g.pstride + i] = P[(size_t)c * g.pstride + nfr * g.N + i];
        if (rc < 0) break;
    }
    free(ws); free(ll); free(bp); free(lfs); free(prs);
    free(bs); free(ts); free(ps); free(B); free(X); free(st);
    return rc;
}
}

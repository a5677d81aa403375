// celt_decoder.cuh — one CELT frame, split along the two pipeline stages.
//
// Restates opus-fix/celt/celt_decoder.c:713-1072 (celt_decode_with_ec):
//   celt_parse_frame  (stage A, scalar)   :833-991  header symbols, coarse/fine energy symbols, tf, spread, dynalloc,
//                                                    trim, compute_allocation, quant_all_bands, anti-collapse bit, finalise
//   celt_synth_frame  (stage B, per team) :842-846,962-964,986-1066  energy prediction, anti_collapse, celt_synthesis
//                                                    (:280-350) with denormalise_bands (bands.c:169-238) fused into the
//                                                    IMDCT pre-rotation, comb_filter (celt.c:156-244), state update,
//                                                    staging for stage C
//   deemphasis_channel (stage C, scalar)  :185-275  de-emphasis + decode gain, one thread per (stream, channel)
#pragma once
#include "celt_bands.cuh"
#include "celt_energy.cuh"
#include "celt_ir.h"
#include "celt_mdct.cuh"
#include "opus_state.h"


namespace cb {

// ---------------------------------------------------------------------------------------------------
// Stage A
// ---------------------------------------------------------------------------------------------------

// Per-thread working set of stage A: a local (stack) object of the parse thread.
struct ParseScratch {
    int16_t norm[2 * 8 * 78];   // folding source
    alignas(16) int16_t tmp[176];           // pulse vector / hadamard staging
    alignas(16) int16_t xw[2 * 176];        // the band being decoded, X | Y: worked on here, copied to the IR once per band
    alignas(16) int16_t lbs[176];           // lowband_scratch
};

// Parse one received CELT frame (payload of `len` >= 2 bytes).  X: C*N int16 for this frame.  *seed is the
// LCG seed on entry (previous frame's final rng) and the frame's final rng on exit.
// dry = true: seed-recovery pass — the identical symbol walk, no spectrum is produced (X, ps untouched).
CB_DEV void celt_parse_frame(const uint8_t *data, int len, int LM, int C, int end, unsigned *seed, CbFrameIR &ir, int16_t *X,
                             ParseScratch &ps, bool dry) {
    const int start = 0;
    const int M = 1 << LM;
    const int N = M * kShortMdct;
    int tf_res[kNbEBands], cap[kNbEBands], offsets[kNbEBands], fine_quant[kNbEBands], pulses[kNbEBands], fine_priority[kNbEBands];
    AllocScratch alloc;
    EcDec dec;
    dec.init(data, (unsigned)len);

    int total_bits = len * 8;
    int tell = dec.tell();
    int silence;
    if (tell >= total_bits) silence = 1;
    else if (tell == 1) silence = dec.bit_logp(15);
    else silence = 0;
    if (silence) {
        tell = len * 8;
        dec.nbits_total += tell - dec.tell();
    }
    int postfilter_gain = 0, postfilter_pitch = 0, postfilter_tapset = 0;
    if (start == 0 && tell + 16 <= total_bits) {
        if (dec.bit_logp(1)) {
            int octave = (int)dec.uint_(6);
            postfilter_pitch = (16 << octave) + (int)dec.bits(4 + octave) - 1;
            int qg = (int)dec.bits(3);
            if (dec.tell() + 2 <= total_bits) postfilter_tapset = dec.icdf(kTapsetIcdf, 2);
            postfilter_gain = 3072 * (qg + 1);   // QCONST16(.09375f,15)
        }
        tell = dec.tell();
    }
    int isTransient = 0;
    if (LM > 0 && tell + 3 <= total_bits) {
        isTransient = dec.bit_logp(3);
        tell = dec.tell();
    }
    const int shortBlocks = isTransient ? M : 0;
    const int intra_ener = tell + 3 <= total_bits ? dec.bit_logp(3) : 0;
    CB_NOUNROLL for (int i = 0; i < 2 * kNbEBands; i++) { ir.qi[i] = 0; ir.eoff[i] = 0; }
    decode_coarse_symbols(start, end, intra_ener, dec, C, LM, ir.qi);
    tf_decode(start, end, isTransient, tf_res, LM, dec);
    tell = dec.tell();
    int spread_decision = kSpreadNormal;
    if (tell + 4 <= total_bits) spread_decision = dec.icdf(kSpreadIcdf, 5);
    init_caps(cap, LM, C);
    int dynalloc_logp = 6;
    total_bits <<= kBitRes;
    tell = (int)dec.tell_frac();
    CB_NOUNROLL for (int i = start; i < end; i++) {
        int width = C * band_width(i) << LM;
        int quanta = imin(width << kBitRes, imax(6 << kBitRes, width));
        int loop_logp = dynalloc_logp;
        int boost = 0;
        while (tell + (loop_logp << kBitRes) < total_bits && boost < cap[i]) {
            int flag = dec.bit_logp(loop_logp);
            tell = (int)dec.tell_frac();
            if (!flag) break;
            boost += quanta;
            total_bits -= quanta;
            loop_logp = 1;
        }
        offsets[i] = boost;
        if (boost > 0) dynalloc_logp = imax(2, dynalloc_logp - 1);
    }
    int alloc_trim = tell + (6 << kBitRes) <= total_bits ? dec.icdf(kTrimIcdf, 7) : 5;
    int bits = ((len * 8) << kBitRes) - (int)dec.tell_frac() - 1;
    int anti_collapse_rsv = isTransient && LM >= 2 && bits >= ((LM + 2) << kBitRes) ? (1 << kBitRes) : 0;
    bits -= anti_collapse_rsv;
    int intensity = 0, dual_stereo = 0, balance = 0;
    AllocDecIo io{dec};
    int codedBands = compute_allocation(io, alloc, start, end, offsets, cap, alloc_trim, &intensity, &dual_stereo, bits, &balance,
                                        pulses, fine_quant, fine_priority, C, LM);
    decode_fine_energy(start, end, fine_quant, dec, C, ir.eoff);

    unsigned sd = *seed;
    quant_all_bands_dec(start, end, X, C == 2 ? X + N : nullptr, ir.collapse, pulses, shortBlocks, spread_decision, dual_stereo,
                        intensity, tf_res, len * (8 << kBitRes) - anti_collapse_rsv, balance, dec, LM, codedBands, &sd, ps.norm,
                        ps.tmp, ps.xw, ps.lbs, dry);
    int anti_collapse_on = 0;
    if (anti_collapse_rsv > 0) anti_collapse_on = (int)dec.bits(1);
    decode_energy_finalise(start, end, fine_quant, fine_priority, len * 8 - dec.tell(), dec, C, ir.eoff);

    ir.rng_final = dec.rng;
    ir.seed_bands = sd;
    ir.len = (int16_t)len;
    ir.pf_pitch = (int16_t)postfilter_pitch;
    ir.pf_gain = (int16_t)postfilter_gain;
    ir.pf_tapset = (uint8_t)postfilter_tapset;
    ir.LM = (uint8_t)LM; ir.C = (uint8_t)C; ir.end = (uint8_t)end;
    ir.flags = (uint8_t)((silence ? CB_IR_SILENCE : 0) | (isTransient ? CB_IR_TRANSIENT : 0) | (intra_ener ? CB_IR_INTRA : 0) |
                         (anti_collapse_on ? CB_IR_ANTICOLLAPSE : 0) | (dec.error ? CB_IR_EC_ERROR : 0) |
                         (dec.tell() > 8 * len ? CB_IR_OVERRUN : 0));
    CB_NOUNROLL for (int i = 0; i < kNbEBands; i++) ir.pulses[i] = (int16_t)(i < end ? pulses[i] : 0);
    *seed = dec.rng;
}

// ---------------------------------------------------------------------------------------------------
// Stage B
// ---------------------------------------------------------------------------------------------------

enum { kDenBins = 100 };   // eBands[nbEBands]: bins of the coded bands at LM = 0

// Team-shared working set of one frame synthesis (~4.8 KB).
struct SynthScratch {
    int fft[kMaxFrame];                               // IMDCT buffer
    int16_t den_gain[2][kNbEBands];                   // denormalisation gain / shift per band
    int8_t den_shift[2][kNbEBands];
    // denormalisation per bin at LM = 0 resolution (bin j of the frame reads den[c][j >> LM]): (G << 5) | R, where
    // X[j] * G >> R equals the reference's gain product and shift (0 outside the decoded bands)
    int den[2][kDenBins];
};

// comb_filter with y == x (celt/celt.c:183-244, as called at celt_decoder.c:1002-1013).  In place the
// filter is recursive: output i reads positions <= i-T+2, already final.  Outputs within a run of
// min(T0,T1)-2 (>= 13) samples are mutually independent, so runs are spread over the lanes.  Every sample it changes is
// also stored to y[i] when y is given.
template <class TM>
CB_DEV void comb_filter_inplace(TM tm, int *x, int T0, int T1, int N, int g0, int g1, int tapset0, int tapset1, int overlap,
                                int *y = nullptr) {
    if (g0 == 0 && g1 == 0) return;
    const int g00 = s16(mul16_16_p15(g0, kCombGains[tapset0][0]));
    const int g01 = s16(mul16_16_p15(g0, kCombGains[tapset0][1]));
    const int g02 = s16(mul16_16_p15(g0, kCombGains[tapset0][2]));
    const int g10 = s16(mul16_16_p15(g1, kCombGains[tapset1][0]));
    const int g11 = s16(mul16_16_p15(g1, kCombGains[tapset1][1]));
    const int g12 = s16(mul16_16_p15(g1, kCombGains[tapset1][2]));
    if (g0 == g1 && T0 == T1 && tapset0 == tapset1) overlap = 0;
    // A tap set whose gain is zero contributes exactly 0 (MULT16_32_Q15(0,.) == 0) whatever its period — the
    // "off" period is 0 in the bitstream — so it is skipped and does not bound the run length.
    const int Tmin = imin(g0 != 0 ? T0 : kCombMaxPeriod, g1 != 0 ? T1 : kCombMaxPeriod);
    const int G = imin(TM::W, Tmin - 2);
    CB_NOUNROLL for (int base = 0; base < overlap; base += G) {
        int i = base + tm.lane();
        if (tm.lane() < G && i < overlap) {
            int f = s16(mul16_16_q15(kWindow120[i], kWindow120[i]));
            int nf = 32767 - f;
            int v = x[i];
            if (g0 != 0) {
                v = wadd(v, mul16_32_q15(mul16_16_q15(nf, g00), x[i - T0]));
                v = wadd(v, mul16_32_q15(mul16_16_q15(nf, g01), wadd(x[i - T0 + 1], x[i - T0 - 1])));
                v = wadd(v, mul16_32_q15(mul16_16_q15(nf, g02), wadd(x[i - T0 + 2], x[i - T0 - 2])));
            }
            if (g1 != 0) {
                v = wadd(v, mul16_32_q15(mul16_16_q15(f, g10), x[i - T1]));
                v = wadd(v, mul16_32_q15(mul16_16_q15(f, g11), wadd(x[i - T1 + 1], x[i - T1 - 1])));
                v = wadd(v, mul16_32_q15(mul16_16_q15(f, g12), wadd(x[i - T1 + 2], x[i - T1 - 2])));
            }
            x[i] = v;
            if (y) y[i] = v;
        }
        tm.sync();
    }
    if (g1 == 0) return;
    CB_NOUNROLL for (int base = overlap; base < N; base += G) {
        int i = base + tm.lane();
        if (tm.lane() < G && i < N) {
            int v = x[i];
            v = wadd(v, mul16_32_q15(g10, x[i - T1]));
            v = wadd(v, mul16_32_q15(g11, wadd(x[i - T1 + 1], x[i - T1 - 1])));
            v = wadd(v, mul16_32_q15(g12, wadd(x[i - T1 + 2], x[i - T1 - 2])));
            x[i] = v;
            if (y) y[i] = v;
        }
        tm.sync();
    }
}

// deemphasis (celt_decoder.c:185-275, accum = 0) is a 1-pole IIR per channel: strictly order dependent, so it is not run
// by the stream's warp (30 idle lanes) but by stage C, one THREAD per (stream, channel), over the staged post-filter
// signal.  x: n samples at 48 kHz; y: int16 PCM with stride CC, decimated by `downsample`; gain = decode gain (Q16, 0 = off,
// opus_decoder.c:567-577).  Returns the filter memory.
CB_DEV int deemphasis_channel(const int *x, int n, int16_t *y, int CC, int downsample, int m, int gain) {
    if (downsample > 1) {
        int k = 0, next = 0;
        CB_NOUNROLL for (int j = 0; j < n; j++) {
            int t = wadd(x[j], m);
            m = mul16_32_q15(kPreemphCoef0, t);
            if (j == next) {
                int v = sig2word16(t);
                if (gain >= 0) { int g = mul16_32_p16(v, gain); v = g > 32767 ? 32767 : (g < -32767 ? -32767 : g); }
                y[k * CC] = (int16_t)v;
                k++;
                next += downsample;
            }
        }
    } else {
        int j = 0;
        // batches of 8 samples: the loads are independent of the recurrence, so they are issued up front (two 16-byte
        // loads when the pointer allows) and the serial chain runs from registers
        if ((((uintptr_t)x) & 15) == 0) {
            CB_NOUNROLL for (; j + 8 <= n; j += 8) {
                int xs[8];
                const int4 a = *reinterpret_cast<const int4 *>(x + j);
                const int4 b = *reinterpret_cast<const int4 *>(x + j + 4);
                xs[0] = a.x; xs[1] = a.y; xs[2] = a.z; xs[3] = a.w; xs[4] = b.x; xs[5] = b.y; xs[6] = b.z; xs[7] = b.w;
#pragma unroll
                CB_NOUNROLL for (int u = 0; u < 8; u++) {
                    int t = wadd(xs[u], m);
                    m = mul16_32_q15(kPreemphCoef0, t);
                    int v = sig2word16(t);
                    if (gain >= 0) { int g = mul16_32_p16(v, gain); v = g > 32767 ? 32767 : (g < -32767 ? -32767 : g); }
                    y[(j + u) * CC] = (int16_t)v;
                }
            }
        }
        CB_NOUNROLL for (; j < n; j++) {
            int t = wadd(x[j], m);
            m = mul16_32_q15(kPreemphCoef0, t);
            int v = sig2word16(t);
            if (gain >= 0) { int g = mul16_32_p16(v, gain); v = g > 32767 ? 32767 : (g < -32767 ? -32767 : g); }
            y[j * CC] = (int16_t)v;
        }
    }
    return m;
}

// Shift the synthesis history down by N samples (celt_decoder.c:962-964), team-parallel and overlap-safe:
// each chunk is read by all lanes before any lane writes it, and destinations trail sources by N >= 120.
template <class TM>
CB_DEV void history_shift(TM tm, int *mem, int N, int count = -1) {
    if (count < 0) count = kDecBuf - N + kOverlap / 2;
    if (((count | N) & 3) == 0) {
        // 16-byte vectors, two per lane and step (the history is 16-byte aligned in the state; N is a multiple of 120)
        int4 *m4 = reinterpret_cast<int4 *>(mem);
        const int nv = count >> 2, sh = N >> 2;
        CB_NOUNROLL for (int base = 0; base < nv; base += 2 * TM::W) {
            const int i0 = base + tm.lane(), i1 = i0 + TM::W;
            int4 a = {0, 0, 0, 0}, b = {0, 0, 0, 0};
            if (i0 < nv) a = m4[i0 + sh];
            if (i1 < nv) b = m4[i1 + sh];
            tm.sync();
            if (i0 < nv) m4[i0] = a;
            if (i1 < nv) m4[i1] = b;
        }
        tm.sync();
        return;
    }
    CB_NOUNROLL for (int base = 0; base < count; base += TM::W) {
        int i = base + tm.lane();
        int v = 0;
        if (i < count) v = mem[i + N];
        tm.sync();
        if (i < count) mem[i] = v;
    }
    tm.sync();
}

// celt_synthesis (celt_decoder.c:280-350) with denormalise_bands (bands.c:169-238) fused into the IMDCT pre-rotation.
// X: C*N normalised spectrum; out_syn[c]: synthesis target (tail of the channel's history).  When sig is given, the
// frame's N output samples of channel c are also stored to sig[c].
template <class TM>
CB_DEV void celt_synthesis_team(TM tm, SynthScratch &S, const int16_t *X, int *const *out_syn, const int16_t *oldBandE, int start, int effEnd,
                                int C, int CC, int isTransient, int LM, int downsample, int silence, int *const *sig = nullptr) {
    const int M = 1 << LM;
    const int N = M * kShortMdct;
    int bstart = start, bend = effEnd;
    int bound = M * kEBands[bend];
    if (downsample != 1) bound = imin(bound, N / downsample);
    if (silence) { bound = 0; bstart = bend = 0; }
    CB_TEAM_FOR(w, C * kNbEBands, tm) {   // per-band gain/shift (bands.c:195-227)
        int c = w / kNbEBands, i = w - c * kNbEBands;
        int lg = s16(oldBandE[c * kNbEBands + i] + shl16(kEMeans[i], 6));
        int shift = 16 - (lg >> 10);
        int g;
        if (shift > 31) { shift = 0; g = 0; }
        else g = celt_exp2_frac(lg & 1023);
        if (shift < -2) { g = 32767; shift = -2; }
        S.den_gain[c][i] = (int16_t)g;
        S.den_shift[c][i] = (int8_t)shift;
    }
    tm.sync();
    // Spread over the bins, with the shift folded into the gain: for shift < 0, (X*g) << -shift == X*(g << -shift)
    // mod 2^32, so each bin costs one multiply and one right shift, without a band look-up or a branch.
    CB_TEAM_FOR(w, C * kDenBins, tm) {
        const int c = w >= kDenBins, k = w - c * kDenBins;
        const int b = kBinToBand[k];
        int e = 0;
        if (b >= bstart && b < bend) {
            const int sh = S.den_shift[c][b];
            e = ((int)S.den_gain[c][b] << (imax(-sh, 0) + 5)) | imax(sh, 0);
        }
        S.den[c][k] = e;
    }
    tm.sync();
    const int B = isTransient ? M : 1;
    const int shift = isTransient ? kMaxLM : kMaxLM - LM;
    const int hi = imin(bound, M * kEBands[bend]);
    auto den = [&](int c, int j) -> int {
        const int e = S.den[c][j >> LM];
        return wmul(X[c * N + j], e >> 5) >> (e & 31);
    };
    // mode 0: channel 0; 1: channel 1; 2: (ch0+ch1)/2 downmix (celt_decoder.c:325-339)
    auto freq = [&](int mode, int j) -> int {
        if (j >= hi) return 0;
        return mode != 2 ? den(mode, j) : (wadd(den(0, j), den(1, j)) >> 1);
    };
    const int npass = (CC == 2 && C == 2) ? 2 : 1;
    CB_NOUNROLL for (int p = 0; p < npass; p++) {
        const int mode = (CC == 1 && C == 2) ? 2 : p;
        imdct_compute(tm, [&](int j) { return freq(mode, j); }, B, shift, S.fft);
        imdct_assemble(tm, out_syn[p], B, shift, S.fft, sig ? sig[p] : nullptr);
        if (CC == 2 && C == 1) imdct_assemble(tm, out_syn[1], B, shift, S.fft, sig ? sig[1] : nullptr);   // mono stream into two channels
    }
}

// Synthesise one received frame from its IR up to (and excluding) de-emphasis: the post-filtered signal of channel c
// (N samples at 48 kHz) is staged to sig[c] for stage C.
// Returns samples per channel at the API rate, or OPUS_INTERNAL_ERROR when the frame overran its bit budget.
template <class TM>
CB_DEV int celt_synth_frame(TM tm, CbDecState *st, SynthScratch &S, const CbFrameIR &ir, int16_t *X, int *const *sig) {
    const int CC = st->channels;
    const int LM = ir.LM, C = ir.C, end = ir.end, start = 0;
    const int M = 1 << LM;
    const int N = M * kShortMdct;
    const int silence = ir.flags & CB_IR_SILENCE, isTransient = (ir.flags & CB_IR_TRANSIENT) != 0;
    int *decode_mem[2], *out_syn[2];
    CB_NOUNROLL for (int c = 0; c < CC; c++) {
        decode_mem[c] = st->decode_mem + c * CB_DEC_MEM;
        out_syn[c] = decode_mem[c] + kDecBuf - N;
    }
    const int effEnd = imin(end, kNbEBands);
    int16_t *oldBandE = st->oldEBands, *oldLogE = st->oldLogE, *oldLogE2 = st->oldLogE2, *backgroundLogE = st->backgroundLogE;

    // ---- energies: the prediction recurrence is serial over bands -> lane 0; the fine offsets are per band ----
    if (tm.lane() == 0) {
        if (C == 1)
            CB_NOUNROLL for (int i = 0; i < kNbEBands; i++) oldBandE[i] = (int16_t)imax(oldBandE[i], oldBandE[kNbEBands + i]);
        apply_coarse_energy(start, end, oldBandE, ir.qi, (ir.flags & CB_IR_INTRA) != 0, C, LM);
    }
    tm.sync();
    CB_TEAM_FOR(w, C * kNbEBands, tm) {
        const int i = w >= kNbEBands ? w - kNbEBands : w;
        if (i >= start && i < end) oldBandE[w] = (int16_t)(oldBandE[w] + ir.eoff[w]);
    }
    tm.sync();
    CB_NOUNROLL for (int c = 0; c < CC; c++) history_shift(tm, decode_mem[c], N);
    if (ir.flags & CB_IR_ANTICOLLAPSE)
        anti_collapse(tm, X, ir.collapse, LM, C, N, start, end, oldBandE, oldLogE, oldLogE2, ir.pulses, ir.seed_bands);
    if (silence) {
        CB_TEAM_FOR(i, C * kNbEBands, tm) oldBandE[i] = -28672;   // -QCONST16(28.f,DB_SHIFT)
        tm.sync();
    }

    // ---- celt_synthesis (celt_decoder.c:280-350) with denormalise_bands (bands.c:169-238) fused in ----
    celt_synthesis_team(tm, S, X, out_syn, oldBandE, start, effEnd, C, CC, isTransient, LM, st->downsample, silence, sig);

    // ---- post-filter (celt_decoder.c:1001-1025); what it changes is staged to sig as well ----
    const int pf_period = imax(st->postfilter_period, kCombMinPeriod);
    const int pf_period_old = imax(st->postfilter_period_old, kCombMinPeriod);
    const int postfilter_pitch = ir.pf_pitch, postfilter_gain = ir.pf_gain, postfilter_tapset = ir.pf_tapset;
    const int max_inc = st->loss_count < 10 ? M : 1024;   // energy history, read before lane 0 resets loss_count: M*QCONST16(0.001f,DB_SHIFT) ; QCONST16(1.f,DB_SHIFT)
    CB_NOUNROLL for (int c = 0; c < CC; c++) {
        comb_filter_inplace(tm, out_syn[c], pf_period_old, pf_period, kShortMdct, st->postfilter_gain_old, st->postfilter_gain,
                            st->postfilter_tapset_old, st->postfilter_tapset, kOverlap, sig[c]);
        if (LM != 0)
            comb_filter_inplace(tm, out_syn[c] + kShortMdct, pf_period, postfilter_pitch, N - kShortMdct, st->postfilter_gain,
                                postfilter_gain, st->postfilter_tapset, postfilter_tapset, kOverlap, sig[c] + kShortMdct);
    }
    tm.sync();
    if (tm.lane() == 0) {
        st->postfilter_period_old = pf_period;
        st->postfilter_gain_old = st->postfilter_gain;
        st->postfilter_tapset_old = st->postfilter_tapset;
        st->postfilter_period = postfilter_pitch;
        st->postfilter_gain = postfilter_gain;
        st->postfilter_tapset = postfilter_tapset;
        if (LM != 0) {
            st->postfilter_period_old = st->postfilter_period;
            st->postfilter_gain_old = st->postfilter_gain;
            st->postfilter_tapset_old = st->postfilter_tapset;
        }
        st->rng = ir.rng_final;
        st->loss_count = 0;
        if (ir.flags & CB_IR_EC_ERROR) st->error = 1;
    }
    // ---- energy history (celt_decoder.c:1027-1062), one band per lane ----
    if (C == 1) {
        CB_TEAM_FOR(i, kNbEBands, tm) oldBandE[kNbEBands + i] = oldBandE[i];
        tm.sync();
    }
    CB_TEAM_FOR(w, 2 * kNbEBands, tm) {
        const int i = w >= kNbEBands ? w - kNbEBands : w;
        const int e = oldBandE[w];
        if (!isTransient) {
            oldLogE2[w] = oldLogE[w];
            oldLogE[w] = (int16_t)e;
            backgroundLogE[w] = (int16_t)imin(backgroundLogE[w] + max_inc, e);
        } else {
            oldLogE[w] = (int16_t)imin(oldLogE[w], e);
        }
        if (i < start || i >= end) {
            oldBandE[w] = 0;
            oldLogE[w] = oldLogE2[w] = -28672;
        }
    }
    tm.sync();
    if (ir.flags & CB_IR_OVERRUN) return OPUS_INTERNAL_ERROR_;
    return N / st->downsample;
}

}  // namespace cb

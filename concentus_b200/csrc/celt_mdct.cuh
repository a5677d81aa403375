// celt_mdct.cuh — fixed-point mixed-radix FFT and the inverse MDCT with TDAC overlap-add.
//
// Restates opus-fix/celt/kiss_fft.c:51-325 (kf_bfly2/4/3/5), :532-578 (opus_fft_impl) and
// celt/mdct.c:263-363 (clt_mdct_backward_c) for the four standard transform sizes
// (N4 = 480/240/120/60 complex points, celt/static_modes_fixed.h:432-499).
//
// Team layout: the FFT buffer (B blocks x N4 complex int32) sits in team-shared memory; inside one
// radix stage all nfft/p butterflies of all B short blocks are independent, so they are strided over
// the lanes with one __syncwarp() per stage.  Stage ORDER and the op order inside a butterfly are
// what fixes the rounding, and both are kept; the order of butterflies within a stage is free.
// The pre-rotation pulls its input through a functor, so band denormalisation (and the stereo->mono
// downmix) is fused into it and the de-normalised spectrum is never materialised.
#pragma once
#include "celt_arith.cuh"
#include "celt_tables.cuh"

namespace cb {

struct Cpx { int r, i; };

CB_DEV int smul(int x, int tw) { return mul16_32_q15(tw, x); }   // S_MUL (_kiss_fft_guts.h:57)
CB_DEV Cpx cmul(Cpx a, int twr, int twi) {                       // C_MUL
    Cpx m;
    m.r = wsub(smul(a.r, twr), smul(a.i, twi));
    m.i = wadd(smul(a.r, twi), smul(a.i, twr));
    return m;
}
CB_DEV Cpx cadd(Cpx a, Cpx b) { Cpx c; c.r = wadd(a.r, b.r); c.i = wadd(a.i, b.i); return c; }
CB_DEV Cpx csub(Cpx a, Cpx b) { Cpx c; c.r = wsub(a.r, b.r); c.i = wsub(a.i, b.i); return c; }
CB_DEV void tw_load(int idx, int &r, int &i) {
    unsigned w = kFftTwiddles[idx];
    r = (int)(int16_t)(w & 0xffff);
    i = (int)(int16_t)(w >> 16);
}

// opus_fft_impl over `nblocks` contiguous transforms of plan `s`.
template <class TM>
CB_DEV void fft_inplace(TM tm, Cpx *buf, int s, int nblocks) {
    const FftPlan &pl = kFftPlan[s];
    const int nfft = pl.nfft;
    CB_NOUNROLL for (int st = 0; st < pl.nstages; st++) {
        const int p = pl.radix[st];
        const int m = pl.m[st];
        const int mm = p * m;
        const int ngroups = nfft / mm;
        const int fs = ngroups << pl.tw_shift;   // twiddle stride (fstride<<shift)
        // Item w = (g, j) with g = block * ngroups + group and j < m.  Blocks are nfft = ngroups * mm apart, so butterfly
        // (g, j) starts at g * mm + j = w + g * (mm - m): one division, by m, and none by ngroups.
        if (p == 2) {
            // kf_bfly2, m == 4 (kiss_fft.c:51-108): item = (block, group, lane-in-group 0..3)
            const int items = nblocks * ngroups * 4;
            CB_TEAM_FOR(w, items, tm) {
                int q = w & 3, g = w >> 2;
                Cpx *F = buf + g * 8 + q;
                Cpx a = F[0], b = F[4], t;
                if (q == 0) t = b;
                else if (q == 1) { t.r = smul(wadd(b.r, b.i), 23170); t.i = smul(wsub(b.i, b.r), 23170); }
                else if (q == 2) { t.r = b.i; t.i = wneg(b.r); }
                else { t.r = smul(wsub(b.i, b.r), 23170); t.i = smul(wsub(wneg(b.i), b.r), 23170); }
                F[4] = csub(a, t);
                F[0] = cadd(a, t);
            }
        } else if (p == 4 && m == 1) {
            // kf_bfly4 degenerate (kiss_fft.c:121-141)
            const int items = nblocks * ngroups;
            CB_TEAM_FOR(w, items, tm) {
                Cpx *F = buf + w * 4;
                Cpx f0 = F[0], f1 = F[1], f2 = F[2], f3 = F[3];
                Cpx s0 = csub(f0, f2);
                f0 = cadd(f0, f2);
                Cpx s1 = cadd(f1, f3);
                f2 = csub(f0, s1);
                f0 = cadd(f0, s1);
                s1 = csub(f1, f3);
                F[0] = f0;
                F[2] = f2;
                Cpx o1, o3;
                o1.r = wadd(s0.r, s1.i); o1.i = wsub(s0.i, s1.r);
                o3.r = wsub(s0.r, s1.i); o3.i = wadd(s0.i, s1.r);
                F[1] = o1;
                F[3] = o3;
            }
        } else if (p == 4) {
            // kf_bfly4 (kiss_fft.c:142-179)
            const int items = nblocks * ngroups * m;
            const unsigned mmag = fastdiv_magic(m);
            CB_TEAM_FOR(w, items, tm) {
                int g = fastdiv(w, mmag), j = w - g * m;
                Cpx *F = buf + w + g * (mm - m);
                int r1, i1, r2, i2, r3, i3;
                tw_load(j * fs, r1, i1);
                tw_load(2 * j * fs, r2, i2);
                tw_load(3 * j * fs, r3, i3);
                Cpx f0 = F[0];
                Cpx c0 = cmul(F[m], r1, i1);
                Cpx c1 = cmul(F[2 * m], r2, i2);
                Cpx c2 = cmul(F[3 * m], r3, i3);
                Cpx c5 = csub(f0, c1);
                f0 = cadd(f0, c1);
                Cpx c3 = cadd(c0, c2);
                Cpx c4 = csub(c0, c2);
                F[2 * m] = csub(f0, c3);
                F[0] = cadd(f0, c3);
                Cpx o1, o3;
                o1.r = wadd(c5.r, c4.i); o1.i = wsub(c5.i, c4.r);
                o3.r = wsub(c5.r, c4.i); o3.i = wadd(c5.i, c4.r);
                F[m] = o1;
                F[3 * m] = o3;
            }
        } else if (p == 3) {
            // kf_bfly3 (kiss_fft.c:185-240), epi3.i = -28378
            const int items = nblocks * ngroups * m;
            const unsigned mmag = fastdiv_magic(m);
            CB_TEAM_FOR(w, items, tm) {
                int g = fastdiv(w, mmag), j = w - g * m;
                Cpx *F = buf + w + g * (mm - m);
                int r1, i1, r2, i2;
                tw_load(j * fs, r1, i1);
                tw_load(2 * j * fs, r2, i2);
                Cpx f0 = F[0];
                Cpx c1 = cmul(F[m], r1, i1);
                Cpx c2 = cmul(F[2 * m], r2, i2);
                Cpx c3 = cadd(c1, c2);
                Cpx c0 = csub(c1, c2);
                Cpx fm;
                fm.r = wsub(f0.r, c3.r >> 1);
                fm.i = wsub(f0.i, c3.i >> 1);
                c0.r = smul(c0.r, -28378);
                c0.i = smul(c0.i, -28378);
                F[0] = cadd(f0, c3);
                Cpx o2, o1;
                o2.r = wadd(fm.r, c0.i); o2.i = wsub(fm.i, c0.r);
                o1.r = wsub(fm.r, c0.i); o1.i = wadd(fm.i, c0.r);
                F[2 * m] = o2;
                F[m] = o1;
            }
        } else {
            // kf_bfly5 (kiss_fft.c:245-318), ya = (10126,-31164), yb = (-26510,-19261)
            const int items = nblocks * ngroups * m;
            const unsigned mmag = fastdiv_magic(m);
            CB_TEAM_FOR(w, items, tm) {
                int g = fastdiv(w, mmag), u = w - g * m;
                Cpx *F = buf + w + g * (mm - m);
                int r1, i1, r2, i2, r3, i3, r4, i4;
                tw_load(u * fs, r1, i1);
                tw_load(2 * u * fs, r2, i2);
                tw_load(3 * u * fs, r3, i3);
                tw_load(4 * u * fs, r4, i4);
                Cpx s0 = F[0];
                Cpx s1 = cmul(F[m], r1, i1);
                Cpx s2 = cmul(F[2 * m], r2, i2);
                Cpx s3 = cmul(F[3 * m], r3, i3);
                Cpx s4 = cmul(F[4 * m], r4, i4);
                Cpx s7 = cadd(s1, s4), s10 = csub(s1, s4);
                Cpx s8 = cadd(s2, s3), s9 = csub(s2, s3);
                Cpx o0;
                o0.r = wadd(s0.r, wadd(s7.r, s8.r));
                o0.i = wadd(s0.i, wadd(s7.i, s8.i));
                F[0] = o0;
                Cpx s5, s6, s11, s12;
                s5.r = wadd(wadd(s0.r, smul(s7.r, 10126)), smul(s8.r, -26510));
                s5.i = wadd(wadd(s0.i, smul(s7.i, 10126)), smul(s8.i, -26510));
                s6.r = wadd(smul(s10.i, -31164), smul(s9.i, -19261));
                s6.i = wsub(wneg(smul(s10.r, -31164)), smul(s9.r, -19261));
                F[m] = csub(s5, s6);
                F[4 * m] = cadd(s5, s6);
                s11.r = wadd(wadd(s0.r, smul(s7.r, -26510)), smul(s8.r, 10126));
                s11.i = wadd(wadd(s0.i, smul(s7.i, -26510)), smul(s8.i, 10126));
                s12.r = wadd(wneg(smul(s10.i, -19261)), smul(s9.i, -31164));
                s12.i = wsub(smul(s10.r, -19261), smul(s9.r, -31164));
                F[2 * m] = cadd(s11, s12);
                F[3 * m] = csub(s11, s12);
            }
        }
        tm.sync();
    }
}

// Inverse MDCT of one channel: B interleaved blocks (coefficient k of block b = freq(b + k*B)),
// overlap-added into `out` (= out_syn of celt_decoder.c:819-821; out[0..overlap/2) holds the tail the
// previous frame left).  shift = maxLM-LM for a long block, maxLM for short blocks.
// Follows mdct.c:263-363 per block; the B blocks' pre-rotation/FFT/post-rotation are batched, then the
// output is assembled in one pass: mirrored (windowed) regions [b*NB, b*NB+overlap) and straight copies.
template <class TM, class FreqFn>
CB_DEV void imdct_compute(TM tm, FreqFn freq, int B, int shift, int *fftbuf) {
    const int N2 = (kMaxFrame * 2 >> shift) >> 1;   // coefficients per block (= NB)
    const int N4 = N2 >> 1;
    int trig_off = 0;
    CB_NOUNROLL for (int i = 0, n = kMaxFrame * 2; i < shift; i++) { n >>= 1; trig_off += n; }
    const int16_t *t = kMdctTwiddles + trig_off;
    const int16_t *bitrev = fft_bitrev(shift);
    const unsigned n4mag = fastdiv_magic(N4), halfmag = fastdiv_magic(N4 >> 1);
    // pre-rotate straight into bit-reversed order (mdct.c:283-303)
    CB_TEAM_FOR(w, B * N4, tm) {
        int b = fastdiv(w, n4mag), i = w - b * N4;
        int x1 = freq(b + (2 * i) * B);
        int x2 = freq(b + (N2 - 1 - 2 * i) * B);
        int t0 = t[i], t1 = t[N4 + i];
        int yr = wadd(smul(x2, t0), smul(x1, t1));
        int yi = wsub(smul(x1, t0), smul(x2, t1));
        int rev = bitrev[i];
        fftbuf[b * N2 + 2 * rev + 1] = yr;
        fftbuf[b * N2 + 2 * rev] = yi;
    }
    tm.sync();
    fft_inplace(tm, (Cpx *)fftbuf, shift, B);
    // post-rotate from both ends (mdct.c:309-343)
    CB_TEAM_FOR(w, B * (N4 >> 1), tm) {   // N4 is even
        int b = fastdiv(w, halfmag), i = w - b * (N4 >> 1);
        int *yp0 = fftbuf + b * N2 + 2 * i;
        int *yp1 = fftbuf + b * N2 + N2 - 2 - 2 * i;
        int re = yp0[1], im = yp0[0];
        int t0 = t[i], t1 = t[N4 + i];
        int yr = wadd(smul(re, t0), smul(im, t1));
        int yi = wsub(smul(re, t1), smul(im, t0));
        re = yp1[1];
        im = yp1[0];
        yp0[0] = yr;
        yp1[1] = yi;
        t0 = t[N4 - i - 1];
        t1 = t[N2 - i - 1];
        yr = wadd(smul(re, t0), smul(im, t1));
        yi = wsub(smul(re, t1), smul(im, t0));
        yp1[0] = yr;
        yp0[1] = yi;
    }
    tm.sync();
}

// Second half of the inverse MDCT: block b produced P_b[k] = fftbuf[b*N2+k], destined for
// out[b*N2 + overlap/2 + k]; positions [b*N2, b*N2+overlap) get the TDAC mirror (mdct.c:346-362).
// The blocks' mirror regions are disjoint and each reads only un-mirrored P values (or, for block 0,
// the tail the previous frame left in out[0..overlap/2)), so the whole output is written in one pass.  When sig is given,
// the frame's samples out[0..N) are also stored to sig[0..N).
template <class TM>
CB_DEV void imdct_assemble(TM tm, int *out, int B, int shift, const int *fftbuf, int *sig = nullptr) {
    const int N2 = (kMaxFrame * 2 >> shift) >> 1;
    const int N = B * N2;
    const int half = kOverlap >> 1;
    const unsigned n2mag = fastdiv_magic(N2);
    CB_TEAM_FOR(j, N + half, tm) {
        int b = fastdiv(j, n2mag);
        int r = j - b * N2;
        if (b < B && r < kOverlap) {
            if (r < half) {
                // pair (i = r): x2 = out_old[b*N2 + i], x1 = out_new[b*N2 + overlap-1-i]
                int i = r;
                int x2 = b == 0 ? out[i] : fftbuf[(b - 1) * N2 + (N2 - half) + i];
                int x1 = fftbuf[b * N2 + (half - 1 - i)];
                int lo = wsub(smul(x2, kWindow120[kOverlap - 1 - i]), smul(x1, kWindow120[i]));
                int hi = wadd(smul(x2, kWindow120[i]), smul(x1, kWindow120[kOverlap - 1 - i]));
                out[b * N2 + i] = lo;
                out[b * N2 + kOverlap - 1 - i] = hi;
                if (sig) {
                    sig[b * N2 + i] = lo;
                    sig[b * N2 + kOverlap - 1 - i] = hi;
                }
            }
        } else {
            // straight copy of P (also the un-mirrored tail [N, N+overlap/2) for the next frame)
            int bb = b < B ? b : B - 1;
            int k = j - bb * N2 - half;
            const int v = fftbuf[bb * N2 + k];
            out[j] = v;
            if (sig && j < N) sig[j] = v;
        }
    }
    tm.sync();
}

// Forward MDCT of one block (mdct.c:121-259): in[N2 + overlap] (windowed fold of the first/last overlap/2 pairs), out with
// `stride` interleave.  f: scratch for N2 ints (fold result), f2: scratch for N2 ints (N4 complex, FFT buffer).
template <class TM>
CB_DEV void mdct_forward(TM tm, const int *in, int *out, int shift, int stride, int *f, int *f2) {
    const int N2 = (kMaxFrame * 2 >> shift) >> 1;
    const int N4 = N2 >> 1;
    int trig_off = 0;
    CB_NOUNROLL for (int i = 0, n = kMaxFrame * 2; i < shift; i++) { n >>= 1; trig_off += n; }
    const int16_t *t = kMdctTwiddles + trig_off;
    const int16_t *bitrev = fft_bitrev(shift);
    const FftPlan &pl = kFftPlan[shift];
    const int scale_shift = pl.scale_shift - 1;
    const int ov = kOverlap, q = (ov + 3) >> 2;
    // window, shuffle, fold (mdct.c:155-203): pair i produces f[2i], f[2i+1]
    CB_TEAM_FOR(i, N4, tm) {
        const int *xp1 = in + (ov >> 1) + 2 * i;
        const int *xp2 = in + N2 - 1 + (ov >> 1) - 2 * i;
        int re, im;
        if (i < q) {
            const int w1 = kWindow120[(ov >> 1) + 2 * i], w2 = kWindow120[(ov >> 1) - 1 - 2 * i];
            re = wadd(smul(xp1[N2], w2), smul(*xp2, w1));
            im = wsub(smul(*xp1, w1), smul(xp2[-N2], w2));
        } else if (i < N4 - q) {
            re = *xp2;
            im = *xp1;
        } else {
            const int k = i - (N4 - q);
            const int w1 = kWindow120[2 * k], w2 = kWindow120[ov - 1 - 2 * k];
            re = wadd(wneg(smul(xp1[-N2], w1)), smul(*xp2, w2));
            im = wadd(smul(*xp1, w2), smul(xp2[N2], w1));
        }
        f[2 * i] = re;
        f[2 * i + 1] = im;
    }
    tm.sync();
    // pre-rotation with scaling into bit-reversed order (mdct.c:205-227)
    CB_TEAM_FOR(i, N4, tm) {
        const int t0 = t[i], t1 = t[N4 + i];
        const int re = f[2 * i], im = f[2 * i + 1];
        int yr = wsub(smul(re, t0), smul(im, t1));
        int yi = wadd(smul(im, t0), smul(re, t1));
        yr = pshr32(mul16_32_q16(kFftScale, yr), scale_shift);
        yi = pshr32(mul16_32_q16(kFftScale, yi), scale_shift);
        const int rev = bitrev[i];
        f2[2 * rev] = yr;
        f2[2 * rev + 1] = yi;
    }
    tm.sync();
    fft_inplace(tm, (Cpx *)f2, shift, 1);
    // post-rotation (mdct.c:233-256)
    CB_TEAM_FOR(i, N4, tm) {
        const int fr = f2[2 * i], fi = f2[2 * i + 1];
        const int yr = wsub(smul(fi, t[N4 + i]), smul(fr, t[i]));
        const int yi = wadd(smul(fr, t[N4 + i]), smul(fi, t[i]));
        out[stride * (2 * i)] = yr;
        out[stride * (N2 - 1 - 2 * i)] = yi;
    }
    tm.sync();
}

}  // namespace cb

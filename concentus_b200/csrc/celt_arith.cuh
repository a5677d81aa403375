// celt_arith.cuh — Q-format integer arithmetic of the FIXED_POINT CELT build, as typed inline functions.
//
// Semantics follow opus-fix/celt/fixed_generic.h:36-151, celt/arch.h:70-118 and celt/mathops.{h,c}
// (reference file:line cited per function).  Conventions used throughout the codec headers:
//   * `int` is the 32-bit working type; a value the reference stores in an opus_val16 is truncated with
//     s16() at exactly the point where the reference assigns/casts it.
//   * 16x32 products are evaluated as one 64-bit product + shift.  This equals the reference's
//     split form ((a*(b>>16))<<1) + ((a*(b&0xffff))>>15) modulo 2^32 because a*(b>>16)*2 is an integer and
//     arithmetic >> is floor — so an IMAD.WIDE + funnel shift replaces six ALU ops.
//   * Signed overflow wraps (two's complement) — all additions that may wrap go through unsigned.
#pragma once
#include "celt_simt.cuh"

namespace cb {

typedef int16_t s16_t;

CB_DEV int s16(int x) { return (int)(int16_t)x; }
CB_DEV int imin(int a, int b) { return a < b ? a : b; }
CB_DEV int imax(int a, int b) { return a > b ? a : b; }
CB_DEV int iabs(int a) { return a < 0 ? -a : a; }
CB_DEV int wadd(int a, int b) { return (int)((unsigned)a + (unsigned)b); }
CB_DEV int wsub(int a, int b) { return (int)((unsigned)a - (unsigned)b); }
CB_DEV int wmul(int a, int b) { return (int)((unsigned)a * (unsigned)b); }
CB_DEV int wneg(int a) { return (int)(0u - (unsigned)a); }

// EC_ILOG (celt/ecintrin.h:67-85): number of bits needed, 0 for x==0 handled by callers.
CB_DEV int ec_ilog(unsigned x) { return 32 - CB_CLZ(x); }

// fixed_generic.h:72-86
CB_DEV int shl32(int a, int s) { return (int)((unsigned)a << s); }
CB_DEV int shr32(int a, int s) { return a >> s; }
CB_DEV int pshr32(int a, int s) { return wadd(a, (1 << s) >> 1) >> s; }
CB_DEV int vshr32(int a, int s) { return s > 0 ? (a >> s) : shl32(a, -s); }
CB_DEV int shl16(int a, int s) { return s16((int)((unsigned)(uint16_t)a << s)); }
CB_DEV int round16(int a, int s) { return s16(pshr32(a, s)); }
CB_DEV int sat16(int x) { return x > 32767 ? 32767 : (x < -32768 ? -32768 : x); }

// fixed_generic.h:113-131 — operands are (truncated to) 16 bit, product is 32 bit.
CB_DEV int mul16_16(int a, int b) { return s16(a) * s16(b); }
CB_DEV int mac16_16(int c, int a, int b) { return wadd(c, s16(a) * s16(b)); }
CB_DEV int mul16_16_q15(int a, int b) { return mul16_16(a, b) >> 15; }
CB_DEV int mul16_16_q14(int a, int b) { return mul16_16(a, b) >> 14; }
CB_DEV int mul16_16_q13(int a, int b) { return mul16_16(a, b) >> 13; }
CB_DEV int mul16_16_q11(int a, int b) { return mul16_16(a, b) >> 11; }
CB_DEV int mul16_16_p15(int a, int b) { return wadd(16384, mul16_16(a, b)) >> 15; }
CB_DEV int mul16_16_p14(int a, int b) { return wadd(8192, mul16_16(a, b)) >> 14; }
CB_DEV int mul16_16_p13(int a, int b) { return wadd(4096, mul16_16(a, b)) >> 13; }

// fixed_generic.h:39-48 (see header note on the 64-bit form).  `a` is a 16-bit value.
CB_DEV int mul16_32_q15(int a, int b) { return (int)(((int64_t)s16(a) * (int64_t)b) >> 15); }
CB_DEV int mul16_32_q16(int a, int b) { return (int)(((int64_t)s16(a) * (int64_t)b) >> 16); }
CB_DEV int mul16_32_p16(int a, int b) { return (int)(((int64_t)s16(a) * (int64_t)b + 32768) >> 16); }
// fixed_generic.h:51 — three partial products, the low x low term is dropped (NOT a 64-bit mul-shift).
CB_DEV int mul32_32_q31(int a, int b) {
    int ah = a >> 16, bh = b >> 16;
    int al = a & 0xffff, bl = b & 0xffff;
    int t0 = shl32(s16(ah) * s16(bh), 1);
    int t1 = (s16(ah) * bl) >> 15;
    int t2 = (s16(bh) * al) >> 15;
    return wadd(wadd(t0, t1), t2);
}
// fixed_generic.h:120 MAC16_32_Q15: b must fit in 31 bits.
CB_DEV int mac16_32_q15(int c, int a, int b) {
    return wadd(c, wadd(s16(a) * s16(b >> 15), (s16(a) * (b & 0x7fff)) >> 15));
}
// FRAC_MUL16 (celt/mathops.h:44)
CB_DEV int frac_mul16(int a, int b) { return (16384 + s16(a) * s16(b)) >> 15; }
// SIG2WORD16 (fixed_generic.h:141-149), SIG_SHIFT = 12
CB_DEV int sig2word16(int x) { return sat16(pshr32(x, 12)); }

// celt_ilog2 / celt_zlog2 (celt/mathops.h:157-170)
CB_DEV int celt_ilog2(int x) { return ec_ilog((unsigned)x) - 1; }
CB_DEV int celt_zlog2(int x) { return x <= 0 ? 0 : celt_ilog2(x); }

// isqrt32 (celt/mathops.c:42-66): exact floor(sqrt(v)).
CB_MATH unsigned isqrt32(unsigned v) {
    unsigned g = 0;
    int bshift = (ec_ilog(v) - 1) >> 1;
    unsigned b = 1u << bshift;
    do {
        unsigned t = ((g << 1) + b) << bshift;
        if (t <= v) { g += b; v -= t; }
        b >>= 1;
        bshift--;
    } while (bshift >= 0);
    return g;
}

// celt_rcp (celt/mathops.c:182-208): Q15 in, Q16 out.
CB_MATH int celt_rcp(int x) {
    int i = celt_ilog2(x);
    int n = s16(vshr32(x, i - 15) - 32768);
    int r = s16(30840 + mul16_16_q15(-15420, n));
    r = s16(r - mul16_16_q15(r, s16(mul16_16_q15(r, n) + s16(r - 32768))));
    r = s16(r - s16(1 + mul16_16_q15(r, s16(mul16_16_q15(r, n) + s16(r - 32768)))));
    return vshr32(r, i - 16);
}
// celt_div (celt/mathops.h:213)
CB_DEV int celt_div(int a, int b) { return mul32_32_q31(a, celt_rcp(b)); }

// frac_div32 (celt/mathops.c:70-91)
CB_MATH int frac_div32(int a, int b) {
    int shift = celt_ilog2(b) - 29;
    a = vshr32(a, shift);
    b = vshr32(b, shift);
    int rcp = round16(celt_rcp(round16(b, 16)), 3);
    int result = mul16_32_q15(rcp, a);
    int rem = wsub(pshr32(a, 2), mul32_32_q31(result, b));
    result = wadd(result, shl32(mul16_32_q15(rcp, rem), 2));
    if (result >= 536870912) return 2147483647;
    if (result <= -536870912) return -2147483647;
    return shl32(result, 2);
}

// celt_rsqrt_norm (celt/mathops.c:94-121): Q16 in [0.25,1), Q14 out.
CB_MATH int celt_rsqrt_norm(int x) {
    int n = s16(x - 32768);
    int r = s16(23557 + mul16_16_q15(n, s16(-13490 + mul16_16_q15(n, 6713))));
    int r2 = s16(mul16_16_q15(r, r));
    int y = shl16(s16(s16(mul16_16_q15(r2, n) + r2)) - 16384, 1);
    return s16(r + mul16_16_q15(r, s16(mul16_16_q15(y, s16(s16(mul16_16_q15(y, 12288)) - 16384)))));
}

// celt_sqrt (celt/mathops.c:124-143)
CB_MATH int celt_sqrt(int x) {
    if (x == 0) return 0;
    if (x >= 1073741824) return 32767;
    int k = (celt_ilog2(x) >> 1) - 7;
    x = vshr32(x, 2 * k);
    int n = s16(x - 32768);
    int rt = s16(23175 + mul16_16_q15(n, s16(11561 + mul16_16_q15(n, s16(-3011 +
              mul16_16_q15(n, s16(1699 + mul16_16_q15(n, -664))))))));
    return vshr32(rt, 7 - k);
}

// _celt_cos_pi_2 / celt_cos_norm (celt/mathops.c:150-179)
CB_MATH int celt_cos_pi_2(int x) {
    int x2 = s16(mul16_16_p15(x, x));
    int inner = wadd(-7651, mul16_16_p15(x2, wadd(8277, mul16_16_p15(-626, x2))));
    int v = wadd((32767 - x2), mul16_16_p15(x2, inner));
    return s16(1 + imin(32766, v));
}
CB_MATH int celt_cos_norm(int x) {
    x = x & 0x0001ffff;
    if (x > (1 << 16)) x = (1 << 17) - x;
    if (x & 0x00007fff) {
        if (x < (1 << 15)) return celt_cos_pi_2(s16(x));
        return s16(-celt_cos_pi_2(s16(65536 - x)));
    }
    if (x & 0x0000ffff) return 0;
    if (x & 0x0001ffff) return -32767;
    return 32767;
}

// celt_log2 (celt/mathops.h:179-193): Q14 in, Q10 out.
CB_MATH int celt_log2(int x) {
    if (x == 0) return -32767;
    int i = celt_ilog2(x);
    int n = s16(vshr32(x, i - 15) - 32768 - 16384);
    int frac = s16(-6793 + mul16_16_q15(n, s16(15746 + mul16_16_q15(n, s16(-5217 +
                mul16_16_q15(n, s16(2545 + mul16_16_q15(n, -1401))))))));
    return s16(shl16(i - 13, 10) + (frac >> 4));
}

// celt_exp2_frac / celt_exp2 (celt/mathops.h:206-225): Q10 in, Q16 out.
CB_DEV int celt_exp2_frac(int x) {
    int frac = shl16(x, 4);
    return s16(16383 + mul16_16_q15(frac, s16(22804 + mul16_16_q15(frac, s16(14819 + mul16_16_q15(10204, frac))))));
}
CB_MATH int celt_exp2(int x) {
    int integer = s16(x) >> 10;
    if (integer > 14) return 0x7f000000;
    if (integer < -15) return 0;
    int frac = celt_exp2_frac(s16(s16(x) - shl16(integer, 10)));
    return vshr32(frac, -integer - 2);
}

// celt_atan01 / celt_atan2p (celt/mathops.h:224-258)
CB_DEV int celt_atan01(int x) {
    return s16(mul16_16_p15(x, wadd(32767, mul16_16_p15(x, wadd(-21, mul16_16_p15(x, wadd(-11943, mul16_16_p15(4936, x))))))));
}
CB_MATH int celt_atan2p(int y, int x) {
    if (y < x) {
        int arg = celt_div(shl32(y, 15), x);
        if (arg >= 32767) arg = 32767;
        return celt_atan01(s16(arg)) >> 1;
    } else {
        int arg = celt_div(shl32(x, 15), y);
        if (arg >= 32767) arg = 32767;
        return 25736 - (celt_atan01(s16(arg)) >> 1);
    }
}

// bitexact_cos / bitexact_log2tan (celt/bands.c:70-94)
CB_MATH int bitexact_cos(int x) {
    x = s16(x);
    int tmp = (4096 + x * x) >> 13;
    int x2 = s16(tmp);
    x2 = s16((32767 - x2) + frac_mul16(x2, (-7651 + frac_mul16(x2, (8277 + frac_mul16(-626, x2))))));
    return s16(1 + x2);
}
CB_MATH int bitexact_log2tan(int isin, int icos) {
    int lc = ec_ilog((unsigned)icos);
    int ls = ec_ilog((unsigned)isin);
    icos <<= 15 - lc;
    isin <<= 15 - ls;
    return (ls - lc) * (1 << 11) + frac_mul16(isin, frac_mul16(isin, -2597) + 7932)
           - frac_mul16(icos, frac_mul16(icos, -2597) + 7932);
}

// celt_lcg_rand (celt/bands.c:63-66)
CB_DEV unsigned lcg_rand(unsigned seed) { return 1664525u * seed + 1013904223u; }
// k steps of the generator at once, k <= 22 (the widest band at LM 0): x -> kLcgMul[k] * x + kLcgAdd[k]  (mod 2^32)
CB_TABLE uint32_t kLcgMul[23] = {1u, 1664525u, 389569705u, 2940799637u, 158984081u, 2862450781u, 3211393721u, 1851289957u, 3934847009u, 2184914861u, 246739401u, 1948736821u, 2941245873u, 4195587069u, 4088025561u, 980655621u, 2001863745u, 657792333u, 65284841u, 1282409429u, 3808694225u, 2968195997u, 2417331449u};
CB_TABLE uint32_t kLcgAdd[23] = {0u, 1013904223u, 1196435762u, 3519870697u, 2868466484u, 1649599747u, 2670642822u, 1476291629u, 2748932008u, 2180890343u, 2498801434u, 3421909937u, 3167820124u, 2636375307u, 3801544430u, 28987765u, 2210837584u, 3039689583u, 1338634754u, 1649346937u, 2768872580u, 2254235155u, 2326606934u};
CB_DEV unsigned lcg_jump(unsigned seed, int k) { return kLcgMul[k] * seed + kLcgAdd[k]; }

// celt_udiv / celt_sudiv are plain divisions in this build (celt/entcode.h:131-160).
CB_DEV unsigned udiv(unsigned n, unsigned d) { return n / d; }
CB_DEV int sudiv(int n, int d) { return n / d; }

// Division of team-loop indices by a divisor fixed for the loop: n / d == umulhi(n, fastdiv_magic(d)) exactly whenever
// 2 <= d and n * d < 2^32 (the rounding error of the magic is below 1/d).  One multiply-high per item instead of the
// dozen-instruction sequence of a division by a runtime value; the magic itself is one division per loop.
CB_DEV unsigned fastdiv_magic(unsigned d) { return 0xffffffffu / d + 1u; }
#if defined(__CUDACC__)
CB_DEV int fastdiv(int n, unsigned magic) { return (int)__umulhi((unsigned)n, magic); }
#else
CB_DEV int fastdiv(int n, unsigned magic) { return (int)(((uint64_t)(unsigned)n * magic) >> 32); }
#endif

}  // namespace cb

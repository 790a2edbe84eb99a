// avdsp_dev.cuh -- device-side arithmetic primitives of the AVDSP executor (sm_100a).
//
// These define the numerics the kernels must reproduce.  Fixed point (DSP_FORMAT 2) is bit-exact
// by construction: int32 x int32 -> int64 products, wrapping 64-bit adds, arithmetic shifts
// (reference: runtime/dsp_fpmath.h, runtime/dsp_biquadSTD.h:25-77).  The float formats follow the
// reference's hand-rolled IEEE helpers (runtime/dsp_ieee754.h) -- truncating multiply, truncating
// int->float, exponent-field shifts -- restated with integer ops so results do not depend on FMA
// contraction or rounding-mode flags.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>
#include "plan.h"

namespace avdsp {

// ---------------------------------------------------------------- fixed point ----------------
// 32x32 -> 64 signed multiply(-accumulate).  How this is spelled decides the SASS (sm_100a, CUDA 12.9):
//   * plain (long long)a * b : NVVM hoists the sign extension of a loop-invariant coefficient out of the loop and
//     the multiply becomes a 64x64 one (IMAD.WIDE.U32 + 2 IMAD + SHF + IADD: 5 instructions per MAC);
//   * inline PTX mad.wide.s32 : ptxas splits chains of them into IMAD.WIDE(.., RZ) products plus 3-input
//     IADD3/IADD3.X carry trees (11 instructions for acc + 5 products);
//   * (long long)a * b on operands passed through an empty volatile asm ("opaque"): NVVM emits
//     mul.wide.s32 + add.s64 and ptxas fuses each pair into ONE accumulating IMAD.WIDE (5 instructions).
// IMAD.WIDE issues at 1/4 rate (measured: 31.6 / clk / SM, tools/microbench_int.cu), so the accumulating form
// is both the fewest issue slots and the fewest fma-pipe cycles.
__device__ __forceinline__ int opaque(int v) { asm volatile("" : "+r"(v)); return v; }
__device__ __forceinline__ long long mul32(int a, int b) { return (long long)opaque(a) * (long long)opaque(b); }
__device__ __forceinline__ long long mac32(long long acc, int a, int b) { return acc + (long long)opaque(a) * (long long)opaque(b); }
// low / high word of a 64-bit value without the trunc/shift patterns NVVM likes to re-widen
__device__ __forceinline__ int lo32(long long v) { int l, h; asm("mov.b64 {%0,%1}, %2;" : "=r"(l), "=r"(h) : "l"(v)); (void)h; return l; }
__device__ __forceinline__ int hi32(long long v) { int l, h; asm("mov.b64 {%0,%1}, %2;" : "=r"(l), "=r"(h) : "l"(v)); (void)l; return h; }
// (int)(acc >> 28): one funnel shift
__device__ __forceinline__ int q59ToS31(long long acc) { return (int)__funnelshift_r((unsigned)lo32(acc), (unsigned)hi32(acc), kMantBQ); }

// dspSaturate64_031 (dsp_fpmath.h:84-98): clamp s4.59 to [-1,1) and return s.31 in the low word
__device__ __forceinline__ long long sat64_031(long long a) {
    const long long lim = 1ll << (kMant + 31);
    if (a >= lim) return 0x7FFFFFFFll;
    if (a < -lim) return (long long)0xFFFFFFFF80000000ull;
    return a >> kMant;
}
// the same as a 32-bit result, decided on the high word only: a >= 2^59 <=> hi >= 2^27, a < -2^59 <=> hi < -2^27
// (one funnel shift + two compare/select pairs instead of two 64-bit comparisons)
__device__ __forceinline__ int sat64_031_s32(long long a) {
    const int lo = lo32(a), hi = hi32(a);
    int v = (int)__funnelshift_r((unsigned)lo, (unsigned)hi, kMant);
    v = hi >= (1 << (kMant - 1)) ? 0x7FFFFFFF : v;
    v = hi < -(1 << (kMant - 1)) ? (int)0x80000000 : v;
    return v;
}

// checkbiquadsat (dsp_biquadSTD.h:25-32): test on the high word only; the negative side clamps one
// high-word step early (hi <= 1-2^27).
__device__ __forceinline__ long long biquadSat(long long acc) {
    const int hi = (int)(acc >> 32);
    const int satpos = 1 << (kMantBQ - 1);
    // in range  <=>  -satpos+2 <= hi <= satpos-1  <=>  (unsigned)(hi + satpos - 2) <= 2*satpos - 3
    if (__builtin_expect((unsigned)(hi + (satpos - 2)) > (unsigned)(2 * satpos - 3), 0)) {
        acc = (hi >= satpos) ? (((long long)satpos << 32) - 1) : -((long long)satpos << 32);
    }
    return acc;
}

// one DF1 biquad section with error feedback (dsp_calc_biquads_int, dsp_biquadSTD.h:34-77).
// state: acc (64-bit, "mantissa reintegration"), x1, x2, y1, y2.  coef: b0 b1 b2 (a1-1) a2 in Q4.28.
struct BqStateI { long long acc; int x1, x2, y1, y2; };
__device__ __forceinline__ int biquadStepI(BqStateI& s, int x, int b0, int b1, int b2, int a1, int a2) {
    long long acc = s.acc;
    acc = mac32(acc, x, b0);
    acc = mac32(acc, s.x1, b1);
    acc = mac32(acc, s.x2, b2);
    acc = mac32(acc, s.y1, a1);
    acc = mac32(acc, s.y2, a2);
    acc = biquadSat(acc);
    s.acc = acc;
    const int y = (int)(acc >> kMantBQ);
    s.x2 = s.x1; s.x1 = x; s.y2 = s.y1; s.y1 = y;
    return y;
}

// ---------------------------------------------------------------- dither PRNG ------------------
// xoshiro128+ (dsp_tpdf.h:35-49) and the TPDF value (dsp_tpdf.h:103-130)
struct Prng { unsigned s0, s1, s2, s3; };
__device__ __forceinline__ unsigned prngNext(Prng& g) {
    const unsigned r = g.s0 + g.s3, t = g.s1 << 9;
    g.s2 ^= g.s0; g.s3 ^= g.s1; g.s1 ^= g.s2; g.s0 ^= g.s3; g.s2 ^= t;
    g.s3 = __funnelshift_l(g.s3, g.s3, 11);
    return r;
}
__device__ __forceinline__ int tpdfDraw(Prng& g, int& white) {
    const int r1 = (int)prngNext(g), r2 = (int)prngNext(g);
    white = r2;
    return (r1 >> 1) + (r2 >> 1);
}
// dspTpdfPrepare (dsp_tpdf.h:55-80)
__host__ __device__ __forceinline__ int ditherMask(int dither)  { return (int)(0xFFFFFFFFu << ((32 - dither) & 31)); }
__host__ __device__ __forceinline__ int ditherShift(int dither) { return kMant - dither + 1; }
__device__ __forceinline__ long long tpdfScaledI(int v, int shift) {       // dspTpdfApply :141-145
    const long long t = v;
    return shift >= 0 ? (long long)((unsigned long long)t << (shift & 63)) : (t >> ((-shift) & 63));
}

// ---------------------------------------------------------------- IEEE helpers -----------------
// dspMulFloatFloat (dsp_ieee754.h:336-375): 24x24 mantissa product, TRUNCATED, inputs/outputs
// flushed to +0 when the (pre-normalisation) exponent underflows.  Exact integer restatement.
static __device__ __forceinline__ float mulFFslow(float a, float b);
// The truncated 24x24 product with the exponent sum IS the IEEE round-toward-zero product whenever the result is a normal
// number that stayed clear of both ends: an exponent field of the hardware result in [2, 253] means the reference's
// pre-normalisation exponent was >= 1 and nothing overflowed (infinite / NaN operands give 255, zero / denormal ones 0, and
// an overflowing product is CLAMPED to the largest finite number by round-toward-zero: field 254).
// Everything else takes the integer restatement.
__device__ __forceinline__ float mulFF(float a, float b) {
    float r; asm("mul.rz.ftz.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
    if (__builtin_expect(((__float_as_uint(r) >> 23) & 255u) - 2u < 252u, 1)) return r;
    return mulFFslow(a, b);
}
static __device__ __forceinline__ float mulFFslow(float a, float b) {
    const unsigned ua = __float_as_uint(a), ub = __float_as_uint(b);
    const int ea = (ua >> 23) & 255, eb = (ub >> 23) & 255;
    if (ea == 0 || eb == 0) return 0.0f;
    int e = ea + eb - 127;
    if (e < 1) return 0.0f;
    if ((ua ^ ub) & 0x80000000u) e |= 256;
    const unsigned long long p = (unsigned long long)((ua & 0x7FFFFFu) | 0x800000u) * ((ub & 0x7FFFFFu) | 0x800000u);
    unsigned hi = (unsigned)(p >> 22);
    if (hi & (1u << 25)) { e++; hi >>= 2; } else hi >>= 1;
    return __uint_as_float((hi & 0x7FFFFFu) | ((unsigned)e << 23));
}
// Fast form of the same product for hot loops: mul.rz.ftz.f32 agrees with mulFF whenever
// ea+eb-127 >= 1 (normal result, no overflow); callers handle the vanishing range themselves.
__device__ __forceinline__ float mulFF_fast(float a, float b) {
    float r; asm("mul.rz.ftz.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b)); return r;
}
// binary32 arithmetic result with the x86 host's NaN rules: an invalid operation gives the negative "real indefinite", a NaN
// operand comes back quieted, the first operand first (the device returns the positive canonical NaN for both)
__device__ __forceinline__ float nanX86(float r, float a, float b) {
    if (__builtin_expect(r == r, 1)) return r;
    const unsigned ua = __float_as_uint(a), ub = __float_as_uint(b);
    if ((ua & 0x7FFFFFFFu) > 0x7F800000u) return __uint_as_float(ua | 0x00400000u);
    if ((ub & 0x7FFFFFFFu) > 0x7F800000u) return __uint_as_float(ub | 0x00400000u);
    return __uint_as_float(0xFFC00000u);
}
// binary32 <-> binary64 conversions and binary64 arithmetic with the x86 host's NaN rules (cvtss2sd / cvtsd2ss keep the sign and the
// top payload bits and set the quiet bit; addsd & co. return the first NaN operand, quieted, and the negative "real indefinite"
// for an invalid operation).  The device's converters return canonical NaNs; a cascade that has blown up to NaN then leaves
// the reference with -1.0 where the device would say +1.0 (the saturation tests the raw sign bit).
__device__ __forceinline__ double f2dX86(float f) {
    if (__builtin_expect(f == f, 1)) return (double)f;
    const unsigned long long u = __float_as_uint(f);
    return __longlong_as_double((long long)(((u & 0x80000000ull) << 32) | 0x7FF8000000000000ull | ((u & 0x003FFFFFull) << 29)));
}
// (tests on the high word: a binary64 compare costs an FP64-pipe instruction, as much as the add it guards)
__device__ __forceinline__ bool d64Special(double d) { return ((unsigned)__double2hiint(d) & 0x7FF00000u) == 0x7FF00000u; }   // inf or NaN
__device__ __forceinline__ bool d64NaN(double d) {
    const unsigned hi = (unsigned)__double2hiint(d);
    return (hi & 0x7FF00000u) == 0x7FF00000u && (((hi & 0x000FFFFFu) | (unsigned)__double2loint(d)) != 0u);
}
__device__ __forceinline__ float d2fX86(double d) {
    if (__builtin_expect(!d64NaN(d), 1)) return (float)d;
    const unsigned long long u = (unsigned long long)__double_as_longlong(d);
    return __uint_as_float((unsigned)((u >> 32) & 0x80000000u) | 0x7FC00000u | (unsigned)((u >> 29) & 0x003FFFFFu));
}
__device__ __forceinline__ double nanX86d(double r, double a, double b) {
    if (__builtin_expect(!d64NaN(r), 1)) return r;
    // (integer tests on the words: the compiler turns a 64-bit mask of the bit pattern into an FP64-pipe |x|)
    if (d64NaN(a)) return __hiloint2double(__double2hiint(a) | 0x00080000, __double2loint(a));
    if (d64NaN(b)) return __hiloint2double(__double2hiint(b) | 0x00080000, __double2loint(b));
    return __hiloint2double((int)0xFFF80000, 0);
}
// ---- exactness guard of the chain kernels' float class ------------------------------------------------------------------
// mul.rz.ftz.f32 IS dspMulFloatFloat except where the reference's integer code leaves IEEE: it flushes on the exponent sum
// BEFORE normalisation (a product in [2^-126, 2^-125) becomes 0) and it knows no overflow (the exponent wraps, where
// round-toward-zero clamps to the largest finite number).  A biquad product is (state value or input) x coefficient, and the
// host admits a program only when every non-zero coefficient lies in [2^-60, 2^7) (chainFloatCoefsInRange).  Then
//  * a product can reach the flush zone only when an operand is a non-zero value below 2^-64: the cascades keep the minimum
//    of the guard word 2*|bits| - 1 (zero maps to the top) over EVERY value they load or produce;
//  * a product can overflow only when an operand is 2^121 or larger, and a step multiplies the largest value by less than
//    2^9.4 (five products of less than 2^7): it is enough to see every sixth step that all values are below 2^64 (the five
//    steps in between stay below 2^111, their products below 2^118) -- the maximum of 2*|bits| on every sixth step (the
//    unroll group); the check also catches infinities and NaNs that came in through the state or the samples.
// Two integer instructions per value (+ one on every sixth step), on the ALU pipe.  A stream that fails either test is
// flagged and re-executed from its state snapshot by the interpreter, whose multiply is the integer restatement (api.cu);
// every value is tested before it can do harm as an operand, so an unflagged stream is the reference's arithmetic bit for bit.
constexpr unsigned kFltGuardTiny = 2u * 0x1F800000u - 1u;          // guard word of 2^-64
constexpr unsigned kFltGuardHuge = 2u * 0x5F800000u;               // 2*|bits| of 2^64
struct FltGuard { unsigned mn = 0xFFFFFFFFu, mx = 0u; };
template <bool HUGE = true>
__device__ __forceinline__ void fltGuard(FltGuard& g, float v) {
    const unsigned b = __float_as_uint(v);
    g.mn = min(g.mn, b + b - 1u);                                  // zero -> 0xFFFFFFFF, tiny -> small
    if (HUGE) g.mx = max(g.mx, b + b);
}
__device__ __forceinline__ bool fltGuardFired(const FltGuard& g) { return g.mn < kFltGuardTiny || g.mx >= kFltGuardHuge; }
// A coefficient from the per-stream table is not checked on the host: one outside [2^-60, 2^7) (non-zero; what
// chainFloatCoefsInRange admits) fires the lane's guard (mn = 0), so the stream is re-executed exactly like one that met a
// tiny value.
__device__ __forceinline__ bool fltCoefOutOfRange(int bits) {
    const unsigned u = (unsigned)bits & 0x7FFFFFFFu, ex = u >> 23;
    return u != 0u && (ex < 127u - 60u || ex > 127u + 6u);
}

// ---- per-stream coefficient table (avdsp_b200_set_coefs) ----------------------------------------------------------------
// The five words b0 b1 b2 a1 a2 of one section: from the table ([column][stream], `col` = the section's b0 column, `pos` = the
// stream's position in the call) when there is one, else from the plan.  Loaded once per launch, before the frame loop.
// Two load paths on purpose: without a table the words stay constant-bank operands of the plan, as they were before tables
// existed (one pointer for both would turn them into generic loads from parameter space).
__device__ __forceinline__ void sectionCoefs(const int* planCf, const int* tab, int pitch, int col, int pos, int c[5]) {
    if (tab) {
        const int* t = tab + (size_t)col * pitch + pos;
#pragma unroll
        for (int q = 0; q < 5; q++) c[q] = __ldg(t + (size_t)q * pitch);
    } else {
#pragma unroll
        for (int q = 0; q < 5; q++) c[q] = planCf[q];
    }
}

// dspMulFloatDouble (:377-410): exact float x float product as a double (zero/denormal inputs -> +0)
__device__ __forceinline__ double mulFD(float a, float b) {
    const unsigned ua = __float_as_uint(a), ub = __float_as_uint(b);
    const int ea = (ua >> 23) & 255, eb = (ub >> 23) & 255;
    if (ea == 0 || eb == 0) return 0.0;
    if (__builtin_expect(ea != 255 && eb != 255, 1)) return __dmul_rn((double)a, (double)b);      // 48-bit product: exact in binary64
    // an infinity or NaN operand (a cascade that blew up): the reference's integer code knows no special values, it adds the
    // exponents, multiplies the mantissas and XORs the signs -- a finite double comes out
    int e = 1023 + ea + eb - 254;
    if ((ua ^ ub) & 0x80000000u) e |= 2048;
    unsigned long long p = (unsigned long long)((ua & 0x7FFFFFu) | 0x800000u) * ((ub & 0x7FFFFFu) | 0x800000u);
    if (p & 0x800000000000ull) { e++; p <<= 5; } else p <<= 6;
    return __longlong_as_double((long long)((p & ((1ull << 52) - 1)) | ((unsigned long long)(long long)e << 52)));
}
// dspIntToFloatScaled (:204-250): truncating conversion, at most 7 right shifts (INT_MIN quirk kept)
__device__ __forceinline__ float i2fScaled(int x, int shift) {
    if (x == 0) return 0.0f;
    int e = 0;
    unsigned acc = (unsigned)x;
    if (x < 0) { acc = 0u - acc; e = 256; }
    const int p = 31 - __clz(acc);
    if (p > 23) { int r = p - 23; if (r > 7) r = 7; acc >>= r; e += r; }
    else        { acc <<= (23 - p); e -= (23 - p); }
    e += 127 + 23 - shift;
    return __uint_as_float((acc & 0x7FFFFFu) | ((unsigned)e << 23));
}
// the same conversion for shift = 31 on the hardware converter: cvt.rz.f32.s32 truncates the magnitude exactly like the
// reference's right shifts for |x| < 2^31, and the scale by 2^-31 is exact; INT_MIN (where the reference's shift cap
// leaves an unnormalised mantissa) takes the restatement
__device__ __forceinline__ float i2f31Fast(int x) {
    if (__builtin_expect(x == (int)0x80000000, 0)) return i2fScaled(x, 31);
    return __fmul_rz(__int2float_rz(x), 4.656612873077393e-10f);
}
// dspIntToDoubleScaled (:252-295): exact
__device__ __forceinline__ double i2dScaled(int x, int shift) {
    if (x == 0) return 0.0;
    int e = 0;
    unsigned acc = (unsigned)x;
    if (x < 0) { acc = 0u - acc; e = 2048; }
    const int p = 31 - __clz(acc);
    acc <<= (31 - p); e -= (31 - p);
    e += 1054 - shift;
    const unsigned long long m = ((unsigned long long)acc << 21) & ((1ull << 52) - 1);
    return __longlong_as_double((long long)(m | ((unsigned long long)(long long)e << 52)));
}
// dsps31Float0DB (:60-83) / dsps31Double0DB (:85-107); shift counts wrap like the x86 build of the
// reference (that is what the oracle pins).
__device__ __forceinline__ int f2s31(float f) {
    const unsigned u = __float_as_uint(f);
    const int e = (u >> 23) & 255;
    if (e == 0) return 0;
    unsigned m = ((u & 0x7FFFFFu) | 0x800000u) << 8;
    const int n = 127 - e;
    if (n > 0) m >>= (n & 31); else m = 0x7FFFFFFFu;
    if (u & 0x80000000u) m = 0u - m;
    return (int)m;
}
// f2s31(satF(f)) for |f| in [2^-31, 1): the mantissa shift is a plain truncation there, i.e. cvt.rzi of f * 2^31 (exact
// scale through the exponent field); everything else (zeros/denormals, |f| >= 1, the x86 shift-count wrap below 2^-31)
// takes the restatement
__device__ __forceinline__ float satF(float f);
__device__ __forceinline__ int f2s31SatFast(int bits) {
    const unsigned e = ((unsigned)bits >> 23) & 255u;
    if (__builtin_expect(e - 96u < 31u, 1)) return __float2int_rz(__int_as_float(bits + (31 << 23)));
    return f2s31(satF(__int_as_float(bits)));
}
__device__ __forceinline__ int d2s31(double d) {
    const unsigned long long u = (unsigned long long)__double_as_longlong(d);
    const int e = (int)((u >> 52) & 2047);
    if (e == 0) return 0;
    long long m = (long long)((u & ((1ull << 52) - 1)) | (1ull << 52));
    const int n = 1044 - e;
    if (n > 21) m >>= (n & 63); else m = 0x7FFFFFFF;
    if ((long long)u < 0) m = -m;
    return (int)m;
}
__device__ __forceinline__ float satF(float f) {                  // dspSaturateFloat0db :170-184
    const int e = ((int)__float_as_uint(f)) >> 23;
    if (e >= 127) return 1.0f;
    if (e < 0 && e >= -129) return -1.0f;
    return f;
}
__device__ __forceinline__ double satD(double d) {                // dspSaturateDouble0db :187-199
    const int e = (int)(__double_as_longlong(d) >> 52);
    if (e >= 1023) return 1.0;
    if (e < 0 && e >= -1025) return -1.0;
    return d;
}
__device__ __forceinline__ float  shiftF(float f, int s)  { return __uint_as_float(__float_as_uint(f) + ((unsigned)s << 23)); }
__device__ __forceinline__ double shiftD(double d, int s) { return __longlong_as_double(__double_as_longlong(d) + (long long)((unsigned long long)(long long)s << 52)); }
__device__ __forceinline__ float truncF(float f, int bit) {       // dspTruncateFloat0DB :112-138
    int i = (int)__float_as_uint(f);
    const int e = (i >> 23) & 255;
    if (e == 0) return 0.0f;
    const int n = 151 - bit - e;
    if (n > 0) {
        if (n >= 24) i = (i >= 0) ? 0 : (int)((unsigned)(256 + 128 - bit) << 23);
        else { const int mask = (int)(0xFFFFFFFFu << n); if (i < 0) i += ~mask; i &= mask; }
    }
    return __uint_as_float((unsigned)i);
}
__device__ __forceinline__ double truncD(double d, int bit) {     // dspTruncateDouble0DB :141-167
    long long i = __double_as_longlong(d);
    const int e = (int)((i >> 52) & 2047);
    if (e == 0) return 0.0;
    const int n = 1076 - bit - e;
    if (n > 0) {
        if (n >= 53) i = (i >= 0) ? 0 : (long long)((unsigned long long)(unsigned)((2048 + 1024 - bit) << 20) << 32);
        else { const long long mask = (long long)(~0ull << n); if (i < 0) i += ~mask; i &= mask; }
    }
    return __longlong_as_double(i);
}

} // namespace avdsp

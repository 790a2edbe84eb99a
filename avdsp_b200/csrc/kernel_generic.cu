// kernel_generic.cu -- generic plan executor: one lane per stream, the whole program per frame.
//
// This is the complete (every opcode, every DSP_FORMAT) path: the B200 replacement of the
// reference's `while(1){switch(opcode)}` interpreter (runtime/dsp_runtime.c:302-1314).  It differs
// from it in three ways: (1) the opcode stream was lowered once on the host (decoder.cpp), so a
// frame only walks resolved micro-ops that sit in the constant bank (the plan is a __grid_constant__
// kernel parameter: micro-op fetches are warp-uniform constant loads); (2) one warp runs 32
// independent streams in lock step, so dispatch is never divergent; (3) all state the reference
// keeps in process globals is per stream.  Programs that consist of independent signal paths take
// the faster systolic kernel (kernel_chain2.cu, kernel_chain3.cu) instead; this one is the always-correct path.
#include "avdsp_dev.cuh"
#include "kernels.h"
#include <algorithm>
#include <cstdlib>

namespace avdsp {

template <int CLS> struct AluT;
template <> struct AluT<ALU_INT64> { typedef long long T; typedef int SP; static constexpr int W = 2; };
template <> struct AluT<ALU_F32>   { typedef float T;     typedef float SP; static constexpr int W = 1; };
template <> struct AluT<ALU_F64>   { typedef double T;    typedef float SP; static constexpr int W = 2; };

// Per-stream state is addressed through a strided pointer: stride 1 when the lane works on its block in HBM, stride
// blockDim when the CTA staged its streams' blocks in shared memory word-interleaved ([word][lane]: conflict-free, and
// no more 32-sector uncoalesced global accesses per state word -- the lanes' blocks are stateWords apart in HBM).
template <typename T> struct SPtr {
    T* p; int s;
    __device__ __forceinline__ SPtr operator+(int k) const { return SPtr{p + (ptrdiff_t)k * s, s}; }
    __device__ __forceinline__ T& operator[](int k) const { return p[(ptrdiff_t)k * s]; }
    __device__ __forceinline__ T& operator*() const { return *p; }
    __device__ __forceinline__ SPtr& operator+=(int k) { p += (ptrdiff_t)k * s; return *this; }
    template <typename U> __device__ __forceinline__ SPtr<U> as() const { return SPtr<U>{reinterpret_cast<U*>(p), s}; }
};
typedef SPtr<int> SPi;

template <int CLS, typename Ptr> __device__ __forceinline__ typename AluT<CLS>::T ldA(Ptr p) {
    if constexpr (CLS == ALU_INT64) return (long long)(((unsigned long long)(unsigned)p[1] << 32) | (unsigned)p[0]);
    else if constexpr (CLS == ALU_F32) return __int_as_float(p[0]);
    else return __longlong_as_double((long long)(((unsigned long long)(unsigned)p[1] << 32) | (unsigned)p[0]));
}
template <int CLS, typename Ptr> __device__ __forceinline__ void stA(Ptr p, typename AluT<CLS>::T v) {
    if constexpr (CLS == ALU_INT64) { p[0] = (int)v; p[1] = (int)(v >> 32); }
    else if constexpr (CLS == ALU_F32) { p[0] = __float_as_int(v); }
    else { const long long b = __double_as_longlong(v); p[0] = (int)b; p[1] = (int)(b >> 32); }
}
template <int CLS, typename Ptr> __device__ __forceinline__ typename AluT<CLS>::SP ldSP(Ptr p) {
    if constexpr (CLS == ALU_INT64) return p[0]; else return __int_as_float(p[0]);
}
template <int CLS, typename Ptr> __device__ __forceinline__ void stSP(Ptr p, typename AluT<CLS>::SP v) {
    if constexpr (CLS == ALU_INT64) p[0] = v; else p[0] = __float_as_int(v);
}
// parameter word -> value
template <int CLS> __device__ __forceinline__ auto par(int bits) {
    if constexpr (CLS == ALU_INT64) return bits; else return __int_as_float(bits);
}
// Plain C arithmetic of the reference's ALU type as its host executes it.  int64: wrapping.  double: the device's binary64 arithmetic
// keeps payloads like the host, its CONVERTERS to and from binary32 do not (avdsp_dev.cuh f2dX86 / d2fX86).  float: the device returns the canonical NaN
// 0x7FFFFFFF for every invalid operation and every NaN input, the x86 host the reference (and the goldens) run on returns the
// "real indefinite" 0xFFC00000 for an invalid operation and the first NaN operand, quieted, otherwise.  That is visible:
// DSP_DITHER in the float formats turns its zero-initialised error word into -inf on the very first frame (dspShiftFloat on
// 0.0, dsp_ieee754.h:297-314), the next frames compute inf - inf, and the saturation (an exponent test on the raw bits,
// :170-184) sends a negative NaN to -1.0 and a positive one to +1.0.
__device__ __forceinline__ long long aAdd(long long a, long long b) { return (long long)((unsigned long long)a + (unsigned long long)b); }
__device__ __forceinline__ long long aSub(long long a, long long b) { return (long long)((unsigned long long)a - (unsigned long long)b); }
__device__ __forceinline__ long long aMul(long long a, long long b) { return (long long)((unsigned long long)a * (unsigned long long)b); }
__device__ __forceinline__ long long aNeg(long long a) { return (long long)(0ull - (unsigned long long)a); }
__device__ __forceinline__ double aAdd(double a, double b) { return nanX86d(__dadd_rn(a, b), a, b); }
__device__ __forceinline__ double aSub(double a, double b) { return nanX86d(__dsub_rn(a, b), a, b); }
__device__ __forceinline__ double aMul(double a, double b) { return nanX86d(__dmul_rn(a, b), a, b); }
__device__ __forceinline__ double aDiv(double a, double b) { return nanX86d(__ddiv_rn(a, b), a, b); }
// ALU value -> float / float -> ALU value as the host converts them
__device__ __forceinline__ float toF(float a) { return a; }
__device__ __forceinline__ float toF(double a) { return d2fX86(a); }
__device__ __forceinline__ float toF(long long a) { return (float)a; }
template <typename T> __device__ __forceinline__ T fromF(float f) { return (T)f; }
template <> __device__ __forceinline__ double fromF<double>(float f) { return f2dX86(f); }
__device__ __forceinline__ double aNeg(double a) { return __longlong_as_double(__double_as_longlong(a) ^ (long long)0x8000000000000000ull); }
__device__ __forceinline__ float aAdd(float a, float b) { return nanX86(__fadd_rn(a, b), a, b); }
__device__ __forceinline__ float aSub(float a, float b) { return nanX86(__fsub_rn(a, b), a, b); }
__device__ __forceinline__ float aMul(float a, float b) { return nanX86(__fmul_rn(a, b), a, b); }
__device__ __forceinline__ float aDiv(float a, float b) { return nanX86(__fdiv_rn(a, b), a, b); }
__device__ __forceinline__ float aNeg(float a) { return __uint_as_float(__float_as_uint(a) ^ 0x80000000u); }      // xorps: flips NaN signs too
__device__ __forceinline__ float aSqrt(float a) {          // sqrt() of the promoted value, rounded back (double rounding is exact for sqrt)
    if (a != a) return __uint_as_float(__float_as_uint(a) | 0x00400000u);
    if (a < 0.0f) return __uint_as_float(0xFFC00000u);
    return __fsqrt_rn(a);
}
__device__ __forceinline__ double aSqrt(double a) { return sqrt(a); }
// cvttss2si: NaN and out-of-range give the "integer indefinite" 0x80000000 (the device would give 0 / saturate)
__device__ __forceinline__ int f2iX86(float f) { return (f >= -2147483648.0f && f < 2147483648.0f) ? (int)f : (int)0x80000000; }

// acc += a*b in the reference's arithmetic (dspmacs64_32_32 / dspMaccFloatFloat)
template <int CLS, typename A, typename B>
__device__ __forceinline__ void macc(typename AluT<CLS>::T& acc, A a, B b) {
    if constexpr (CLS == ALU_INT64) acc = mac32(acc, a, b);
    else if constexpr (CLS == ALU_F32) acc = aAdd(acc, mulFF(a, b));
    else acc = aAdd(acc, mulFD(a, b));
}
template <int CLS> __device__ __forceinline__ typename AluT<CLS>::T i2a(int v, int shift) {
    if constexpr (CLS == ALU_F32) return i2fScaled(v, shift);
    else if constexpr (CLS == ALU_F64) return i2dScaled(v, shift);
    else return (long long)v;
}

struct TpdfTab { int dither, mask, shift; };
__device__ __forceinline__ TpdfTab makeTab(int d) { TpdfTab t; t.dither = d; t.mask = ditherMask(d); t.shift = ditherShift(d); return t; }

template <int CLS>
__device__ __forceinline__ void tpdfApply(typename AluT<CLS>::T& X, const TpdfTab& t, int tpdfValue) {
    if constexpr (CLS == ALU_INT64) X += tpdfScaledI(tpdfValue, t.shift);
    else if constexpr (CLS == ALU_F32) X = aAdd(X, i2fScaled(tpdfValue, 31 + t.dither - 1));
    else X = aAdd(X, i2dScaled(tpdfValue, 31 + t.dither - 1));
}
template <int CLS>
__device__ __forceinline__ void tpdfTruncate(typename AluT<CLS>::T& X, const TpdfTab& t) {
    if constexpr (CLS == ALU_INT64) X &= (long long)((unsigned long long)(long long)t.mask << kMant);
    else if constexpr (CLS == ALU_F32) X = truncF(X, t.dither);
    else X = truncD(X, t.dither);
}
template <int CLS>
__device__ __forceinline__ typename AluT<CLS>::T saturate(typename AluT<CLS>::T X) {
    if constexpr (CLS == ALU_INT64) return sat64_031(X);
    else if constexpr (CLS == ALU_F32) return satF(X);
    else return satD(X);
}

struct StreamRegs { Prng g; int tpdfValue, tpdfRandom, dither; };
// this stream's view of the per-stream tables (GenericArgs::coefs, ::firTaps), nullptr where the instance has none: its word of
// biquad column c is coefs[c * pitch], its tap of FIR column c is fir[c]; firCol: the column of micro-op i's first tap
struct CoefRow { const int* coefs; int pitch, step; const int* fir; const int* firCol; };

// Execute ops[i0,i1) of one core for one frame.  `io` is this lane's 32-slot sample array in shared
// memory (stride = blockDim.x), `st` its state block in HBM.
template <int CLS, bool TAB>
__device__ __forceinline__ void runCore(const GenericPlan& P, int i0, int i1, int* __restrict__ io, const int ios,
                                        const SPi st, const int* __restrict__ big, StreamRegs& R, const CoefRow crow) {
    typedef typename AluT<CLS>::T ALU;
    typedef typename AluT<CLS>::SP SPT;
    constexpr int AW = AluT<CLS>::W;
    ALU X = 0, Y = 0;
    TpdfTab tp = makeTab(R.dither);                // dsp_runtime.c:306-307: every core call starts on the global table
    bool tpLocal = false;                          // true once DSP_TPDF switched this core to a local table
    const bool sampleInt = P.h.sampleInt != 0;
#define IO(slot) io[(slot) * ios]
    for (int i = i0; i < i1; i++) {
        const MicroOp m = P.ops[i];
        switch (m.op) {
        case OP_SWAPXY: { ALU t = X; X = Y; Y = t; break; }
        case OP_COPYXY: Y = X; break;
        case OP_COPYYX: X = Y; break;
        case OP_CLRXY:  X = 0; Y = 0; break;
        case OP_ADDXY: X = aAdd(X, Y); break;
        case OP_ADDYX: Y = aAdd(Y, X); break;
        case OP_SUBXY: X = aSub(X, Y); break;
        case OP_SUBYX: Y = aSub(Y, X); break;
        case OP_NEGX:  X = aNeg(X); break;
        case OP_NEGY:  Y = aNeg(Y); break;
        case OP_MULXY: X = aMul(X, Y); break;
        case OP_DIVXY:
            if constexpr (CLS == ALU_INT64) X = (Y == 0 || (X == LLONG_MIN && Y == -1)) ? 0 : X / Y; else X = aDiv(X, Y);
            break;
        case OP_DIVYX:
            if constexpr (CLS == ALU_INT64) Y = (X == 0 || (Y == LLONG_MIN && X == -1)) ? 0 : Y / X; else Y = aDiv(Y, X);
            break;
        case OP_AVGXY: if constexpr (CLS == ALU_INT64) X = X / 2 + Y / 2; else X = aAdd(aDiv(X, (ALU)2), aDiv(Y, (ALU)2)); break;
        case OP_AVGYX: if constexpr (CLS == ALU_INT64) Y = X / 2 + Y / 2; else Y = aAdd(aDiv(X, (ALU)2), aDiv(Y, (ALU)2)); break;
        case OP_SHIFT:
            if constexpr (CLS == ALU_INT64) {
                const int n = m.a;
                if (n >= 0) X = (long long)((unsigned long long)X << ((n >= 100 ? kMant : n) & 63));
                else        X = X >> ((n <= -100 ? kMant : -n) & 63);
            } else if constexpr (CLS == ALU_F32) X = shiftF(X, m.a);
            else X = shiftD(X, m.a);
            break;
        case OP_SQRTX:
            if constexpr (CLS == ALU_INT64) {
                unsigned res = 0;
                if (X >> 32) {
                    for (unsigned bit = 1u << 30; bit; bit >>= 1) { const unsigned t = res | bit; if (X >= (long long)((unsigned long long)t * t)) res = t; }
                } else {
                    for (unsigned bit = 1u << 15; bit; bit >>= 1) { unsigned t = res | bit; t *= t; if (X >= (long long)t) res = t; }
                }
                X = res;
            } else X = aSqrt(X);
            break;
        case OP_SAT0DB: X = saturate<CLS>(X); break;
        case OP_SAT0DB_TPDF: tpdfApply<CLS>(X, tp, R.tpdfValue); X = saturate<CLS>(X); break;
        case OP_SAT0DB_GAIN: case OP_SAT0DB_TPDF_GAIN: {
            if constexpr (CLS == ALU_INT64) { X >>= kMant; X = X * (long long)m.a; }
            else if constexpr (CLS == ALU_F32) X = mulFF(X, __int_as_float(m.a));
            else X = mulFD(toF(X), __int_as_float(m.a));
            if (m.op == OP_SAT0DB_TPDF_GAIN) tpdfApply<CLS>(X, tp, R.tpdfValue);
            X = saturate<CLS>(X);
            break; }
        case OP_TPDF_CALC: {
            if (m.a == R.dither) {
                R.tpdfValue = tpdfDraw(R.g, R.tpdfRandom);
                X = i2a<CLS>(R.tpdfValue, 31);
                stA<CLS>(st + m.b, X);
            } else {                                 // table rebuilt, no PRNG step (dsp_runtime.c:539-544)
                R.dither = m.a;
                if (!tpLocal) tp = makeTab(m.a);     // this core is (still) using the global table
                X = 0;
            }
            break; }
        case OP_TPDF: {
            if (m.a != tp.dither) { tp = makeTab(m.a); tpLocal = true; }   // core-local table (dsp_runtime.c:549)
            X = i2a<CLS>(R.tpdfValue, 31);
            stA<CLS>(st + m.b, X);
            break; }
        case OP_WHITE: X = i2a<CLS>(R.tpdfRandom, 31); break;
        case OP_LOAD:
            Y = X;
            if constexpr (CLS == ALU_INT64) X = IO(m.a);
            else X = sampleInt ? i2a<CLS>(IO(m.a), 31) : fromF<ALU>(__int_as_float(IO(m.a)));
            break;
        case OP_LOAD_GAIN:
            Y = X;
            if constexpr (CLS == ALU_INT64) X = mul32(IO(m.a), m.b);
            else if (sampleInt) {
                const float t = i2fScaled(IO(m.a), 31);
                if constexpr (CLS == ALU_F32) X = mulFF(t, __int_as_float(m.b)); else X = mulFD(t, __int_as_float(m.b));
            } else { X = fromF<ALU>(__int_as_float(IO(m.a))); X = aMul(X, (ALU)__int_as_float(m.b)); }
            break;
        case OP_LOAD_MUX: {
            X = 0;
            for (int k = 0; k < m.n; k++) {
                const int slot = P.pool[m.a + 2 * k], g = P.pool[m.a + 2 * k + 1];
                if constexpr (CLS == ALU_INT64) macc<CLS>(X, IO(slot), g);
                else { const float s = sampleInt ? i2fScaled(IO(slot), 31) : __int_as_float(IO(slot)); macc<CLS>(X, s, __int_as_float(g)); }
            }
            stA<CLS>(st + m.b, X);
            break; }
        case OP_STORE:
            if constexpr (CLS == ALU_INT64) IO(m.a) = (int)X & tp.mask;
            else if (sampleInt) { if constexpr (CLS == ALU_F32) IO(m.a) = f2s31(X) & tp.mask; else IO(m.a) = d2s31(X) & tp.mask; }
            else IO(m.a) = __float_as_int(toF(X));
            break;
        case OP_LOAD_STORE:
            for (int k = 0; k < m.n; k++) IO(P.pool[m.a + 2 * k + 1]) = IO(P.pool[m.a + 2 * k]);
            break;
        case OP_LOAD_MEM:      Y = X; X = ldA<CLS>(st + m.a); break;
        case OP_STORE_MEM:     stA<CLS>(st + m.a, X); break;
        case OP_LOAD_MEM_DATA: X = ldA<CLS>(st + m.a); break;
        case OP_GAIN: case OP_MUL_VALUE:
            if constexpr (CLS == ALU_INT64) X = X * (long long)m.a; else X = aMul(X, (ALU)__int_as_float(m.a));
            break;
        case OP_VALUE: Y = X; if constexpr (CLS == ALU_INT64) X = m.a; else X = (ALU)__int_as_float(m.a); break;
        case OP_VALUE_INT: Y = X; X = (ALU)m.a; break;
        case OP_MUL_VALUE_INT: X = aMul(X, (ALU)m.a); break;
        case OP_DIV_VALUE:
            if constexpr (CLS == ALU_INT64) X = (m.a == 0) ? 0 : X / m.a; else X = aDiv(X, (ALU)__int_as_float(m.a));
            break;
        case OP_DIV_VALUE_INT:
            if constexpr (CLS == ALU_INT64) X = (m.a == 0) ? 0 : X / m.a; else X = aDiv(X, (ALU)m.a);
            break;
        case OP_AND_VALUE_INT:
            if constexpr (CLS == ALU_INT64) X &= (long long)m.a;
            break;
        case OP_DELAY_1: { Y = X; const ALU t = ldA<CLS>(st + m.a); stA<CLS>(st + m.a, X); X = t; break; }
        case OP_DELAY: {
            SPi d = st + m.a;
            int idx = d[0];
            const SPT old = ldSP<CLS>(d + 1 + idx);
            if constexpr (CLS == ALU_INT64) stSP<CLS>(d + 1 + idx, (SPT)X); else stSP<CLS>(d + 1 + idx, toF(X));
            X = old;
            idx++; if ((unsigned)idx >= (unsigned)m.b) idx = 0;
            d[0] = idx;
            break; }
        case OP_DELAY_DP: {
            SPi d = st + m.a;
            int idx = d[0];
            const ALU old = ldA<CLS>(d + 1 + idx * AW);
            stA<CLS>(d + 1 + idx * AW, X);
            X = old;
            idx++; if ((unsigned)idx >= (unsigned)m.b) idx = 0;
            d[0] = idx;
            break; }
        case OP_BIQUADS: {
            SPi s = st + m.a;
            // the plan's coefficients, or this stream's row of the coefficient table: column m.c, then coefStep per section
            const bool tab = TAB && crow.coefs;
            const int* cf = tab ? crow.coefs + (size_t)m.c * crow.pitch : P.pool + m.b;
            const size_t cq = tab ? (size_t)crow.pitch : 1, cs = tab ? (size_t)crow.step * crow.pitch : 5;
            if constexpr (CLS == ALU_INT64) {
                int xn = (int)(X >> kMantBQ);
                long long acc = 0;
                for (int k = 0; k < m.n; k++, s += 6, cf += cs) {
                    BqStateI q; q.acc = ldA<CLS>(s); q.x1 = s[2]; q.x2 = s[3]; q.y1 = s[4]; q.y2 = s[5];
                    xn = biquadStepI(q, xn, cf[0], cf[cq], cf[2 * cq], cf[3 * cq], cf[4 * cq]);
                    acc = q.acc;
                    stA<CLS>(s, q.acc); s[2] = q.x1; s[3] = q.x2; s[4] = q.y1; s[5] = q.y2;
                }
                X = acc;
            } else {
                float xn = toF(X);
                ALU acc = 0;
                for (int k = 0; k < m.n; k++, s += 6, cf += cs) {
                    acc = ldA<CLS>(s);
                    const float x1 = __int_as_float(s[2]), x2 = __int_as_float(s[3]);
                    const float y1 = __int_as_float(s[4]), y2 = __int_as_float(s[5]);
                    macc<CLS>(acc, xn, __int_as_float(cf[0]));
                    macc<CLS>(acc, x1, __int_as_float(cf[cq]));
                    macc<CLS>(acc, x2, __int_as_float(cf[2 * cq]));
                    macc<CLS>(acc, y1, __int_as_float(cf[3 * cq]));
                    macc<CLS>(acc, y2, __int_as_float(cf[4 * cq]));
                    stA<CLS>(s, acc);
                    s[2] = __float_as_int(xn); s[3] = __float_as_int(x1); s[5] = __float_as_int(y1);
                    xn = toF(acc);
                    s[4] = __float_as_int(xn);
                }
                X = acc;
            }
            break; }
        case OP_FIR: {
            SPi s = st + m.a;
            if (m.n == 0) {                                   // plain delay of m.b samples, stores X>>28
                // dsp_runtime.c:943 reads/writes the ring index through the dspALU_SP_t pointer: a float in formats 3..6
                int idx;
                if constexpr (CLS == ALU_INT64) idx = s[0]; else idx = (int)__int_as_float(s[0]);
                const SPT old = ldSP<CLS>(s + 1 + idx);
                if constexpr (CLS == ALU_INT64) s[1 + idx] = (int)(X >> kMant); else stSP<CLS>(s + 1 + idx, toF(X));
                X = old;
                idx++; if (idx >= m.b) idx = 0;
                if constexpr (CLS == ALU_INT64) s[0] = idx; else s[0] = __float_as_int((float)idx);
            } else {
                // the plan's taps, or this stream's row of the FIR table (from the column of this micro-op)
                const int* taps = (TAB && crow.fir) ? crow.fir + __ldg(crow.firCol + i) : big + m.b;
                if constexpr (CLS == ALU_INT64) {            // intended semantics, see DESIGN.md "FIR"
                    int xn = (int)(X >> kMantBQ);
                    long long acc = 0;
                    for (int k = 0; k < m.c; k++) { const int prev = s[k]; s[k] = xn; acc = mac32(acc, xn, taps[k]); xn = prev; }
                    X = acc;
                } else {                                     // dsp_calc_fir_float (dsp_firSTD.h:38-52)
                    float xn = toF(X);
                    ALU acc = 0;
                    for (int k = 0; k < m.c; k++) {
                        const float prev = __int_as_float(s[k]); s[k] = __float_as_int(xn);
                        macc<CLS>(acc, xn, __int_as_float(taps[k]));
                        xn = prev;
                    }
                    X = acc;
                }
            }
            break; }
        case OP_DATA_TABLE: {
            const int* q = P.pool + m.a;                      // gain, div, size, idxOff, tableOff
            SPi ip = st + q[3];
            int idx = *ip;
            const int raw = big[q[4] + idx];
            idx += q[1]; if (idx >= q[2]) idx -= q[2];
            *ip = idx;
            if constexpr (CLS == ALU_INT64) X = mul32(raw, q[0]);
            else {
                const float sv = sampleInt ? (float)raw : __int_as_float(raw);
                if constexpr (CLS == ALU_F32) X = mulFF(sv, __int_as_float(q[0])); else X = mulFD(sv, __int_as_float(q[0]));
            }
            break; }
        case OP_DCBLOCK: {
            SPi ap = st + m.a; SPi sp = ap + AW;
            if constexpr (CLS == ALU_INT64) {
                int xn = (int)(X >> kMant);
                const int prevX = sp[0]; sp[0] = xn;
                xn = (int)((unsigned)xn - (unsigned)prevX);
                X = ldA<CLS>(ap);
                const int prevY = sp[1];
                X = mac32(X, xn, 1 << kMant);
                X = mac32(X, prevY, m.b);
                stA<CLS>(ap, X);
                sp[1] = (int)(X >> kMant);
            } else {
                float xn = toF(X);
                const float prevX = __int_as_float(sp[0]); sp[0] = __float_as_int(xn);
                xn = aSub(xn, prevX);
                X = ldA<CLS>(ap);
                const float prevY = toF(X);
                X = aAdd(X, fromF<ALU>(xn));
                macc<CLS>(X, prevY, __int_as_float(m.b));
                stA<CLS>(ap, X);
            }
            break; }
        case OP_DITHER: {
            SPi e = st + m.a;
            ALU t0 = ldA<CLS>(e); const ALU t1 = ldA<CLS>(e + AW), t2 = ldA<CLS>(e + 2 * AW);
            X = aAdd(X, t0);
            if constexpr (CLS == ALU_INT64) t0 >>= 1; else if constexpr (CLS == ALU_F32) t0 = shiftF(t0, -1); else t0 = shiftD(t0, -1);
            X = aSub(X, t1); X = aAdd(X, t2);
            stA<CLS>(e + AW, t0); stA<CLS>(e + 2 * AW, t1);
            const ALU s0 = X;
            tpdfApply<CLS>(X, tp, R.tpdfValue); tpdfTruncate<CLS>(X, tp);
            stA<CLS>(e, aSub(s0, X));
            break; }
        case OP_DITHER_NS2: {
            SPi e = st + m.a;
            const SPT e0 = ldSP<CLS>(e), e1 = ldSP<CLS>(e + 1), e2 = ldSP<CLS>(e + 2);
            macc<CLS>(X, e0, par<CLS>(P.pool[m.b]));
            macc<CLS>(X, e1, par<CLS>(P.pool[m.b + 1]));
            macc<CLS>(X, e2, par<CLS>(P.pool[m.b + 2]));
            stSP<CLS>(e + 1, e0); stSP<CLS>(e + 2, e1);
            ALU s0 = X;
            tpdfApply<CLS>(X, tp, R.tpdfValue); tpdfTruncate<CLS>(X, tp);
            s0 = aSub(s0, X);
            if constexpr (CLS == ALU_INT64) e[0] = (int)(s0 >> kMant); else stSP<CLS>(e, (SPT)s0);
            break; }
        case OP_RMS: {
            SPtr<unsigned> d = (st + m.a).as<unsigned>();
            const unsigned delay = (unsigned)m.b;
            const unsigned counter = d[0] + 1;
            const unsigned maxCounter = (unsigned)P.pool[m.c];
            const int factor = P.pool[m.c + 1];
            SPi sumsq = (d + 5).as<int>(); SPi avg = sumsq + AW;
            if constexpr (CLS == ALU_INT64) {
                if (factor > 0) { const int sv = (int)(((long long)(int)X * factor) >> 32); X = ldA<CLS>(sumsq); X = mac32(X, sv, sv); }
                else { const int sx = (int)(((long long)(int)X * factor) >> 32), sy = (int)(((long long)(int)Y * factor) >> 32);
                       X = ldA<CLS>(sumsq); X = mac32(X, sx, sy); }
            } else { if (factor > 0) X = aMul(X, X); else X = aMul(X, Y); X = aAdd(X, ldA<CLS>(sumsq)); }
            if (counter >= maxCounter) {
                if (delay) {
                    unsigned idx = d[1];
                    SPi line = sumsq + (2 * AW + (int)idx * AW);
                    const ALU old = ldA<CLS>(line);
                    stA<CLS>(line, X);
                    X = aSub(X, old); X = aAdd(X, ldA<CLS>(avg));
                    idx++; if (idx >= delay) idx = 0;
                    d[1] = idx;
                }
                stA<CLS>(avg, X);
                d[0] = 0;
                stA<CLS>(sumsq, (ALU)0);
                X = (ALU)d[2];
            } else {
                stA<CLS>(sumsq, X);
                d[0] = counter;
                if constexpr (CLS == ALU_INT64) {
                    if (counter == 1) { d[4] = 1u << 30; d[3] = 0; X = (long long)d[2]; }
                    else {
                        const unsigned bit = d[4];
                        if (bit) {
                            const unsigned t = d[3] | bit;
                            if (ldA<CLS>(avg) >= (long long)((unsigned long long)t * t)) d[3] = t;
                            d[4] = bit >> 1;
                            X = (long long)d[2];
                        } else { X = (long long)d[3]; d[2] = (unsigned)X; }
                    }
                } else X = aSqrt(ldA<CLS>(avg));
            }
            break; }
        case OP_DISTRIB: {
            const int size = m.b;
            SPi d = st + m.c; SPi tab = d + 1;
            int idx = d[0];
            const int middle = size >> 1;
            SPT sv;
            if constexpr (CLS == ALU_INT64) sv = (SPT)X; else sv = toF(X);
            if (sv != 0) {
                int pos;
                if constexpr (CLS == ALU_INT64) pos = (int)(((long long)sv * size) >> 32); else pos = f2iX86(aMul(sv, (float)middle));
                pos += middle;
                if (pos >= 0 && pos < size) tab[pos]++;
            }
            int v = tab[idx];
            if (v == 0) v = idx ? tab[idx - 1] : tab[1];
            idx++; if (idx >= size) idx = 0;
            d[0] = idx;
            if constexpr (CLS == ALU_INT64) IO(m.a) = v;
            else IO(m.a) = sampleInt ? v : __float_as_int(i2fScaled(v, 31));
            break; }
        case OP_DIRAC: case OP_SQUAREWAVE: {
            SPi cp = st + m.a;
            int counter = *cp;
            if (m.op == OP_DIRAC) {
                if (counter == 0) { if constexpr (CLS == ALU_INT64) X = mul32(0x7FFFFFFF, m.b); else X = (ALU)__int_as_float(m.b); }
            } else {
                const bool hi = counter <= (m.c / 2);
                if constexpr (CLS == ALU_INT64) X = mul32(hi ? 0x40000000 : (int)0xC0000000, m.b);
                else if constexpr (CLS == ALU_F32) X = mulFF(hi ? 0.5f : -0.5f, __int_as_float(m.b));
                else X = mulFD(hi ? 0.5f : -0.5f, __int_as_float(m.b));
            }
            counter++; if (counter >= m.c) counter = 0;
            *cp = counter;
            break; }
        case OP_CLIP: {
            ALU th;
            if constexpr (CLS == ALU_INT64) th = (long long)((unsigned long long)0x80000000u * (unsigned long long)(unsigned)m.a);
            else th = (ALU)__int_as_float(m.a);
            if (X > th) X = th; else if (X < aNeg(th)) X = aNeg(th);
            break; }
        default: break;
        }
    }
#undef IO
}

// TAB: the launch reads a per-stream biquad coefficient table (GenericArgs::coefs), a per-stream FIR table (::firTaps) or both.
// A template argument rather than a test: the interpreter reads coefficients every frame, and the plan-only instance stays
// what it was without the tables.
template <int CLS, bool TAB>
__global__ void __launch_bounds__(kGenericThreads)
k_generic(const __grid_constant__ GenericPlan P, const GenericArgs A) {
    extern __shared__ int io_s[];                       // [kIoSlots][blockDim.x], then (staged) [stateWords][blockDim.x]
    const int ios = blockDim.x;
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= A.nStreams) return;
    if (A.redo && !A.redo[s]) return;                   // second pass behind a float chain kernel: flagged streams only
    int* io = io_s + threadIdx.x;
    int* gst = A.state + (size_t)s * P.h.stateWords;
    // longer launches work on a shared-memory copy of the state blocks ([word][lane]); each lane moves its own block
    const bool staged = A.stageState != 0;
    const SPi st = staged ? SPi{io_s + kIoSlots * ios + threadIdx.x, ios} : SPi{gst, 1};
    const int* src = A.redo ? A.snapshot + (size_t)s * P.h.stateWords : gst;
    if (staged) for (int w = 0; w < P.h.stateWords; w++) st[w] = src[w];
    else if (A.redo) for (int w = 0; w < P.h.stateWords; w++) gst[w] = src[w];
    const SPi aux = st + P.h.auxOff;
    StreamRegs R;
    R.g.s0 = aux[AUX_S0]; R.g.s1 = aux[AUX_S1]; R.g.s2 = aux[AUX_S2]; R.g.s3 = aux[AUX_S3];
    R.tpdfValue = aux[AUX_TPDF_VALUE]; R.tpdfRandom = aux[AUX_TPDF_RANDOM]; R.dither = aux[AUX_DITHER];
    const int* in = A.in + (size_t)s * A.inStreamStride;
    int* out = A.out + (size_t)s * A.outStreamStride;
    const CoefRow crow{TAB && A.coefs ? A.coefs + s : nullptr, A.coefPitch, A.coefStep,
                       TAB && A.firTaps ? A.firTaps + (size_t)s * A.firPitch : nullptr, A.firCol};
    const int c0 = A.coreSel >= 0 ? A.coreSel : 0;
    const int c1 = A.coreSel >= 0 ? A.coreSel + 1 : P.h.nCores;

    if (A.period <= 0) {
        // canonical order: frame-major, cores ascending, one io[] per frame shared by all cores
        for (int f = 0; f < A.nFrames; f++) {
#pragma unroll
            for (int k = 0; k < kIoSlots; k++) io[k * ios] = 0;
            for (int k = 0; k < P.h.nIn; k++) io[P.h.inIdx[k] * ios] = in[(size_t)f * A.inFrameStride + (size_t)k * A.inChStride];
            for (int c = c0; c < c1; c++) runCore<CLS, TAB>(P, P.h.coreStart[c], P.h.coreStart[c + 1], io, ios, st, A.bigPool, R, crow);
            for (int k = 0; k < P.h.nOut; k++) out[(size_t)f * A.outFrameStride + (size_t)k * A.outChStride] = io[P.h.outIdx[k] * ios];
        }
    } else {
        // ALSA plugin order (linux/avdsp_plugin.c:95-142): core-major inside each period, fresh io[] per
        // (core, frame); outputs a core does not own keep what an earlier core wrote.
        for (int base = 0; base < A.nFrames; base += A.period) {
            const int cnt = min(A.period, A.nFrames - base);
            for (int c = c0; c < c1; c++)
                for (int f = base; f < base + cnt; f++) {
#pragma unroll
                    for (int k = 0; k < kIoSlots; k++) io[k * ios] = 0;
                    for (int k = 0; k < P.h.nIn; k++)
                        if ((A.coreInMask[c] >> P.h.inIdx[k]) & 1u) io[P.h.inIdx[k] * ios] = in[(size_t)f * A.inFrameStride + (size_t)k * A.inChStride];
                    runCore<CLS, TAB>(P, P.h.coreStart[c], P.h.coreStart[c + 1], io, ios, st, A.bigPool, R, crow);
                    for (int k = 0; k < P.h.nOut; k++)
                        if ((A.coreOutMask[c] >> P.h.outIdx[k]) & 1u) out[(size_t)f * A.outFrameStride + (size_t)k * A.outChStride] = io[P.h.outIdx[k] * ios];
                }
        }
    }
    const SPi auxw = st + P.h.auxOff;
    auxw[AUX_S0] = R.g.s0; auxw[AUX_S1] = R.g.s1; auxw[AUX_S2] = R.g.s2; auxw[AUX_S3] = R.g.s3;
    auxw[AUX_TPDF_VALUE] = R.tpdfValue; auxw[AUX_TPDF_RANDOM] = R.tpdfRandom; auxw[AUX_DITHER] = R.dither;
    if (staged) for (int w = 0; w < P.h.stateWords; w++) gst[w] = st[w];
}

cudaError_t launchGeneric(const GenericPlan& plan, const GenericArgs& args, cudaStream_t stream) {
    GenericArgs A = args;
    int threads = A.nStreams >= 4 * kGenericThreads ? kGenericThreads : 32;
    // stage the state blocks in shared memory when the launch is long enough to pay for the two copies and a warp's
    // blocks fit: as many threads per CTA as ~96 KB allow (more CTAs per SM beat wider CTAs: the lanes are latency-bound)
    A.stageState = 0;
    const size_t perLane = (size_t)(kIoSlots + plan.h.stateWords) * sizeof(int);
    if (A.nFrames >= 32 && perLane * 32 <= 200 * 1024 && !getenv("AVDSP_B200_GENERIC_NO_STAGE")) {
        A.stageState = 1;
        int t = (int)((96 * 1024) / perLane) / 32 * 32;
        threads = std::max(32, std::min(threads, t));
    }
    const int blocks = (A.nStreams + threads - 1) / threads;
    const size_t smem = (size_t)threads * (A.stageState ? perLane : kIoSlots * sizeof(int));
    cudaError_t e = cudaSuccess;
#define LAUNCH_G1(CLS, TAB) do { \
        e = cudaFuncSetAttribute(k_generic<CLS, TAB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(smem, 48 * 1024)); \
        if (e != cudaSuccess) return e; \
        k_generic<CLS, TAB><<<blocks, threads, smem, stream>>>(plan, A); } while (0)
#define LAUNCH_G(CLS) do { if (A.coefs || A.firTaps) LAUNCH_G1(CLS, true); else LAUNCH_G1(CLS, false); } while (0)
    switch (plan.h.aluClass) {
    case ALU_INT64: LAUNCH_G(ALU_INT64); break;
    case ALU_F32:   LAUNCH_G(ALU_F32); break;
    default:        LAUNCH_G(ALU_F64); break;
    }
#undef LAUNCH_G
#undef LAUNCH_G1
    return cudaGetLastError();
}

} // namespace avdsp

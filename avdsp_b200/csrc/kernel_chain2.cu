// kernel_chain2.cu -- warp-specialised systolic executor for programs made of independent signal paths
//     source (LOAD / LOAD_GAIN / LOAD_MUX) -> biquad cascade -> [GAIN] -> SAT0DB[_TPDF][_GAIN] -> [DELAY] -> STORE
// (crossovers, EQs: configs C2, C3).  Fixed point (DSP_FORMAT 2), bit-exact.
//
// Why it looks like this (B200: 148 SMs; the signed 32x32+64 IMAD.WIDE issues at 1/4 rate = 31.6 / clk / SM
// measured, everything else at 1 instruction / clk / SMSP):
//   * The biquad recurrence is sequential in time, so time stays a loop.  Parallelism = streams x paths x
//     sections.  A *section lane* owns K consecutive sections of one cascade: state (64-bit accumulator,
//     x1 x2 y1 y2; reference layout runtime/dsp_biquadSTD.h:45) and the 5 Q4.28 coefficients stay in
//     registers for the whole launch.  The cascade is skewed in time ("systolic"): at step t the section
//     with index g inside its cascade works on frame t-g, so all sections of a step are independent
//     (ILP inside a lane, one __shfl_up between lanes) -- exact, because section g of frame n only needs
//     section g-1 of the same frame (dsp_calc_biquads_int, runtime/dsp_biquadSTD.h:37-74).
//   * A section costs 5 accumulating IMAD.WIDE = 20 fma-pipe cycles per warp; the lane-step around K=2 of them
//     is 26 issue slots (SASS checked), so the section warps are fma-pipe bound and leave ~1/3 of the issue
//     slots to the rest.  Nothing else is allowed into that loop: tiles are fully unrolled, shared-memory
//     offsets are immediates, rings are indexed by STEP (identical position for every lane; the per-cascade
//     skew is absorbed by the helpers), the saturation test is one vote + branch per lane-step.
//   * Everything else is element-wise over (stream, frame) and is done by *helper warps* of the same CTA,
//     one tile ahead (TMA-staged PCM -> sources -> x ring) and one tile behind (accumulator ring -> gain /
//     saturate / dither -> post ring; post ring -> delay -> mask -> 16-byte stores).  Helper warp 0 advances the
//     per-stream dither PRNG (xoshiro128+, strictly serial per stream: one lane per stream).  Helper code keeps
//     off the fma pipe: addresses are sums of host-precomputed byte offsets (constant-bank operands).
//     Roles meet only at tile boundaries through named barriers (bar.arrive / bar.sync).
//   * One CTA per SM owns NS = ceil(nStreams / #SM) streams for the whole launch; state never leaves the
//     SM between tiles.  4096 streams -> 147 CTAs x 28 streams, single wave.
//
// Ring bookkeeping (F = tile length, g_c = cascade length - 1 = frame lag of cascade c's tail, gmax <= F):
//   x ring    [stream][source][2F]  by step: head lanes read position t for frame t
//   acc ring  [stream][row][2F]     by step: tail of cascade c writes at step t the accumulator of frame t-g_c
//                                   (only cascades followed by gain / dither; a cascade -> SAT0DB tail writes its y1
//                                   straight into the post ring)
//   post ring [slot][R]             by step: saturated s.31 value of the same frame; R >= 2F+gmax+longest delay (power
//                                   of two): it doubles as the delay line, so steady state never touches HBM state
//   tpdf ring [stream][4F]          by frame (helper warp 0 may run one tile ahead of the others)
//   sink window i = frames [iF-gmax, (i+1)F-gmax): every cascade has finished them when tile i is done.
#include "avdsp_dev.cuh"
#include "kernels.h"
#include <algorithm>
#include <cstdlib>
#include <vector>

namespace avdsp {

constexpr int kBarFull = 1;       // +parity : x tile ready            (helpers arrive, sections wait)
constexpr int kBarDone = 3;       // +parity : section tile finished   (sections arrive, helpers wait)
#ifndef AVDSP_UNR
#define AVDSP_UNR 8
#endif
constexpr int UNR = AVDSP_UNR;    // section steps unrolled per loop iteration (must divide the tile length)

__device__ __forceinline__ void barSync(int id, int n)   { asm volatile("bar.sync %0, %1;" :: "r"(id), "r"(n) : "memory"); }
__device__ __forceinline__ void barArrive(int id, int n) { asm volatile("bar.arrive %0, %1;" :: "r"(id), "r"(n) : "memory"); }

// ---- shared memory by 32-bit address (no generic-pointer arithmetic in the hot paths)
__device__ __forceinline__ unsigned smemAddr(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ int lds32(unsigned a) { int v; asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(a) : "memory"); return v; }
__device__ __forceinline__ long long lds64(unsigned a) { long long v; asm volatile("ld.shared.b64 %0, [%1];" : "=l"(v) : "r"(a) : "memory"); return v; }
__device__ __forceinline__ void sts32(unsigned a, int v) { asm volatile("st.shared.b32 [%0], %1;" :: "r"(a), "r"(v) : "memory"); }

// ---- TMA (1-D bulk copy global -> shared, completion on an mbarrier): how input PCM tiles reach the SM
__device__ __forceinline__ void mbarInit(unsigned bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbarExpectTx(unsigned bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tmaLoad1D(unsigned dst, const void* src, unsigned bytes, unsigned bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void mbarWait(unsigned bar, unsigned parity) {
    asm volatile("{\n"
                 ".reg .pred P1;\n"
                 "LAB_WAIT:\n"
                 "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
                 "@P1 bra DONE;\n"
                 "bra LAB_WAIT;\n"
                 "DONE:\n"
                 "}" :: "r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void fenceProxyAsync() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

template <int K>
struct Lane2 {
    long long acc[K];
    int x1[K], x2[K], y1[K], y2[K];
    int b0[K], b1[K], b2[K], a1[K], a2[K];
};

constexpr unsigned kSatBias  = (1u << (kMantBQ - 1)) - 2u;       // in range  <=>  (unsigned)(hi + bias) <= limit
constexpr unsigned kSatLimit = (1u << kMantBQ) - 3u;             // (checkbiquadsat, runtime/dsp_biquadSTD.h:25-32)

// one lane-step, all K sections valid, OPTIMISTIC: no saturation handling, only a sticky record of the largest
// biased high word seen (checkbiquadsat, runtime/dsp_biquadSTD.h:25-32, fires iff that record exceeds kSatLimit).
// The caller tests the record once per tile and, in the rare case it fired, replays the tile from a checkpoint
// with laneStepExact.  (A vote + branch per step costs ~25 % of the loop: branches and VOTE are not free next to
// a quarter-rate IMAD.WIDE stream, tools/microbench_mix.cu.)
template <int K>
__device__ __forceinline__ void laneStepFast(Lane2<K>& L, int xin, unsigned& worst) {
    int in[K];
    in[0] = xin;
#pragma unroll
    for (int j = 1; j < K; j++) in[j] = L.y1[j - 1];          // skew: section j takes what j-1 produced one step ago
#pragma unroll
    for (int j = 0; j < K; j++) {
        long long acc = L.acc[j];
        acc = mac32(acc, L.x1[j], L.b1[j]);
        acc = mac32(acc, L.x2[j], L.b2[j]);
        acc = mac32(acc, L.y1[j], L.a1[j]);
        acc = mac32(acc, L.y2[j], L.a2[j]);
        acc = mac32(acc, in[j], L.b0[j]);
        worst = max(worst, (unsigned)hi32(acc) + kSatBias);
        L.acc[j] = acc;
        L.x2[j] = L.x1[j]; L.x1[j] = in[j];
        L.y2[j] = L.y1[j]; L.y1[j] = q59ToS31(acc);
    }
}
// the same lane-step with the reference's saturation applied to every section
template <int K>
__device__ __forceinline__ void laneStepExact(Lane2<K>& L, int xin) {
    int in[K];
    in[0] = xin;
#pragma unroll
    for (int j = 1; j < K; j++) in[j] = L.y1[j - 1];
#pragma unroll
    for (int j = 0; j < K; j++) {
        long long acc = L.acc[j];
        acc = mac32(acc, L.x1[j], L.b1[j]);
        acc = mac32(acc, L.x2[j], L.b2[j]);
        acc = mac32(acc, L.y1[j], L.a1[j]);
        acc = mac32(acc, L.y2[j], L.a2[j]);
        acc = mac32(acc, in[j], L.b0[j]);
        acc = biquadSat(acc);
        L.acc[j] = acc;
        L.x2[j] = L.x1[j]; L.x1[j] = in[j];
        L.y2[j] = L.y1[j]; L.y1[j] = q59ToS31(acc);
    }
}

// lane-step at the edges of the launch: section j commits only when its frame t-g0-j lies in [0,T)
template <int K>
__device__ __forceinline__ void laneStepPred(Lane2<K>& L, int xin, int t, int g0, int T) {
    int in[K];
    in[0] = xin;
#pragma unroll
    for (int j = 1; j < K; j++) in[j] = L.y1[j - 1];
#pragma unroll
    for (int j = 0; j < K; j++) {
        if ((unsigned)(t - g0 - j) < (unsigned)T) {
            long long acc = L.acc[j];
            acc = mac32(acc, L.x1[j], L.b1[j]);
            acc = mac32(acc, L.x2[j], L.b2[j]);
            acc = mac32(acc, L.y1[j], L.a1[j]);
            acc = mac32(acc, L.y2[j], L.a2[j]);
            acc = mac32(acc, in[j], L.b0[j]);
            acc = biquadSat(acc);
            L.acc[j] = acc;
            L.x2[j] = L.x1[j]; L.x1[j] = in[j];
            L.y2[j] = L.y1[j]; L.y1[j] = q59ToS31(acc);
        }
    }
}

// ---- DSP_FORMAT 3 (float ALU, int32 samples): dsp_calc_biquads_float, runtime/dsp_biquadSTD.h:84-119.
// acc += x*b0; += x1*b1; += x2*b2; += y1*(a1); += y2*a2 in THIS order, every product truncated
// (dspMulFloatFloat, runtime/dsp_ieee754.h:336-375 == mul.rz.ftz.f32 except when the product underflows next to
// 2^-126, where the reference flushes one binade earlier: an error of at most 2^-125, 95 bits below the s.31
// LSB -- the stated tolerance of this kernel; tests require identical s.31 output), every sum rounded to nearest.
// No saturation inside a float cascade.
template <int K>
struct Lane2F {
    float acc[K], x1[K], x2[K], y1[K], y2[K];
    float b0[K], b1[K], b2[K], a1[K], a2[K];
};
template <int K, bool HUGE = true>
__device__ __forceinline__ void laneStepF(Lane2F<K>& L, float xin, FltGuard& mn) {
    float in[K];
    in[0] = xin;
#pragma unroll
    for (int j = 1; j < K; j++) in[j] = L.y1[j - 1];
#pragma unroll
    for (int j = 0; j < K; j++) {
        float acc = L.acc[j];
        acc = __fadd_rn(acc, mulFF_fast(in[j], L.b0[j]));
        acc = __fadd_rn(acc, mulFF_fast(L.x1[j], L.b1[j]));
        acc = __fadd_rn(acc, mulFF_fast(L.x2[j], L.b2[j]));
        acc = __fadd_rn(acc, mulFF_fast(L.y1[j], L.a1[j]));
        acc = __fadd_rn(acc, mulFF_fast(L.y2[j], L.a2[j]));
        fltGuard<HUGE>(mn, acc);
        L.acc[j] = acc;
        L.x2[j] = L.x1[j]; L.x1[j] = in[j];
        L.y2[j] = L.y1[j]; L.y1[j] = acc;
    }
}
// K = 2 interior steps with the two sections of the lane packed into f32x2 operands (sm_100a: FMUL2.FTZ.RZ / FADD2): the
// same per-element arithmetic in half the issue slots -- the float lane-step is issue-bound, not FP32-pipe-bound.
struct Lane2FP { unsigned long long acc, x1, x2, y1, y2, b0, b1, b2, a1, a2; };
__device__ __forceinline__ unsigned long long packF2(float lo, float hi) { unsigned long long r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ float loF2(unsigned long long v) { float lo, hi; asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); (void)hi; return lo; }
__device__ __forceinline__ float hiF2(unsigned long long v) { float lo, hi; asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); (void)lo; return hi; }
__device__ __forceinline__ unsigned long long macF2(unsigned long long acc, unsigned long long a, unsigned long long b) {
    unsigned long long p;
    asm("mul.rz.ftz.f32x2 %0, %1, %2;" : "=l"(p) : "l"(a), "l"(b));
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(acc) : "l"(acc), "l"(p));
    return acc;
}
__device__ __forceinline__ void packLane(const Lane2F<2>& L, Lane2FP& Q) {
    Q.acc = packF2(L.acc[0], L.acc[1]); Q.x1 = packF2(L.x1[0], L.x1[1]); Q.x2 = packF2(L.x2[0], L.x2[1]);
    Q.y1 = packF2(L.y1[0], L.y1[1]); Q.y2 = packF2(L.y2[0], L.y2[1]);
    Q.b0 = packF2(L.b0[0], L.b0[1]); Q.b1 = packF2(L.b1[0], L.b1[1]); Q.b2 = packF2(L.b2[0], L.b2[1]);
    Q.a1 = packF2(L.a1[0], L.a1[1]); Q.a2 = packF2(L.a2[0], L.a2[1]);
}
__device__ __forceinline__ void unpackLane(const Lane2FP& Q, Lane2F<2>& L) {
    L.acc[0] = loF2(Q.acc); L.acc[1] = hiF2(Q.acc); L.x1[0] = loF2(Q.x1); L.x1[1] = hiF2(Q.x1); L.x2[0] = loF2(Q.x2); L.x2[1] = hiF2(Q.x2);
    L.y1[0] = loF2(Q.y1); L.y1[1] = hiF2(Q.y1); L.y2[0] = loF2(Q.y2); L.y2[1] = hiF2(Q.y2);
}
template <bool HUGE>
__device__ __forceinline__ void laneStepFP(Lane2FP& Q, float xin, FltGuard& mn) {
    const unsigned long long in = packF2(xin, loF2(Q.y1));           // section 1 works on section 0's previous output
    unsigned long long acc = Q.acc;
    acc = macF2(acc, in, Q.b0);
    acc = macF2(acc, Q.x1, Q.b1);
    acc = macF2(acc, Q.x2, Q.b2);
    acc = macF2(acc, Q.y1, Q.a1);
    acc = macF2(acc, Q.y2, Q.a2);
    fltGuard<HUGE>(mn, loF2(acc)); fltGuard<HUGE>(mn, hiF2(acc));
    Q.acc = acc;
    Q.x2 = Q.x1; Q.x1 = in;
    Q.y2 = Q.y1; Q.y1 = acc;
}

// EXACT (second pass over flagged streams): dspMulFloatFloat as hardware product + integer fallback, the host's NaN rules on the sums
template <bool EXACT> __device__ __forceinline__ float maccF2(float acc, float a, float b) {
    if (EXACT) return nanX86(__fadd_rn(acc, mulFF(a, b)), acc, mulFF(a, b));
    return __fadd_rn(acc, mulFF_fast(a, b));
}
template <int K, bool EXACT = false>
__device__ __forceinline__ void laneStepPredF(Lane2F<K>& L, float xin, int t, int g0, int T, FltGuard& mn) {
    float in[K];
    in[0] = xin;
#pragma unroll
    for (int j = 1; j < K; j++) in[j] = L.y1[j - 1];
#pragma unroll
    for (int j = 0; j < K; j++) {
        if ((unsigned)(t - g0 - j) < (unsigned)T) {
            float acc = L.acc[j];
            acc = maccF2<EXACT>(acc, in[j], L.b0[j]);
            acc = maccF2<EXACT>(acc, L.x1[j], L.b1[j]);
            acc = maccF2<EXACT>(acc, L.x2[j], L.b2[j]);
            acc = maccF2<EXACT>(acc, L.y1[j], L.a1[j]);
            acc = maccF2<EXACT>(acc, L.y2[j], L.a2[j]);
            if (!EXACT) fltGuard(mn, acc);
            L.acc[j] = acc;
            L.x2[j] = L.x1[j]; L.x1[j] = in[j];
            L.y2[j] = L.y1[j]; L.y1[j] = acc;
        }
    }
}
// float-class source from GLOBAL memory: dsp_runtime.c:565-607, 871-897.  DSP_FORMAT 3: int32 samples (dspIntToFloatScaled, LOAD_GAIN
// through dspMulFloatFloat); DSP_FORMAT 5: the sample IS the float and LOAD_GAIN is a plain C multiply
__device__ __forceinline__ float sampleF(int smp, bool sampleInt) { return sampleInt ? i2fScaled(smp, 31) : __int_as_float(smp); }
__device__ __forceinline__ float chainSourceF(const ChainPlan& P, const ChainDesc& d, const int* __restrict__ in, int chStride) {
    const bool si = P.h.sampleInt != 0;
    if (d.srcKind == SRC_LOAD_MUX) {
        float X = 0.0f;
        for (int k = 0; k < d.srcCh; k++) {
            const int ch = P.pool[d.srcArg + 2 * k], gain = P.pool[d.srcArg + 2 * k + 1];
            { const float p_ = mulFF(sampleF(ch >= 0 ? in[(size_t)ch * chStride] : 0, si), __int_as_float(gain)); X = nanX86(__fadd_rn(X, p_), X, p_); }
        }
        return X;
    }
    const float t = sampleF(d.srcCh >= 0 ? in[(size_t)d.srcCh * chStride] : 0, si);
    if (d.srcKind != SRC_LOAD_GAIN) return t;
    const float g = __int_as_float(d.srcArg);
    return si ? mulFF(t, g) : nanX86(__fmul_rn(t, g), t, g);
}
// float-class post-processing of one accumulator: [GAIN] -> SAT0DB[_GAIN][_TPDF] (dsp_runtime.c:464-534, 636-640)
__device__ __forceinline__ float finishF(float X, int flags, int gainBits, int satGainBits, int tv, int dither) {
    if (flags & PF_GAIN) { const float g = __int_as_float(gainBits); X = nanX86(__fmul_rn(X, g), X, g); }       // a C multiply: the host's NaN rules
    if (flags & PF_SAT_GAIN) X = mulFF(X, __int_as_float(satGainBits));
    if (flags & PF_SAT_TPDF) { const float d_ = i2fScaled(tv, 31 + dither - 1); X = nanX86(__fadd_rn(X, d_), X, d_); }
    return satF(X);
}

// source value of a chain for one frame from GLOBAL memory: LOAD / LOAD_GAIN / LOAD_MUX (dsp_runtime.c:565-607, 871-897)
__device__ __forceinline__ long long chainSource(const ChainPlan& P, const ChainDesc& d, const int* __restrict__ in, int chStride) {
    if (d.srcKind == SRC_LOAD_MUX) {
        long long X = 0;
        for (int k = 0; k < d.srcCh; k++) {
            const int ch = P.pool[d.srcArg + 2 * k], gain = P.pool[d.srcArg + 2 * k + 1];
            X = mac32(X, ch >= 0 ? in[(size_t)ch * chStride] : 0, gain);
        }
        return X;
    }
    const int smp = d.srcCh >= 0 ? in[(size_t)d.srcCh * chStride] : 0;
    return (d.srcKind == SRC_LOAD_GAIN) ? mul32(smp, d.srcArg) : (long long)smp;
}
// LOAD_MUX from a TMA-staged tile (shared address of channel 0 of the frame, channel stride in bytes)
__device__ __forceinline__ long long muxFromShared(const ChainPlan& P, const ChainDesc& d, unsigned a, unsigned chBytes) {
    long long X = 0;
    for (int k = 0; k < d.srcCh; k++) {
        const int ch = P.pool[d.srcArg + 2 * k], gain = P.pool[d.srcArg + 2 * k + 1];
        X = mac32(X, ch >= 0 ? lds32(a + ch * chBytes) : 0, gain);
    }
    return X;
}

// cascade -> DELAY -> SAT0DB*: the ring value is the low word of a Q59 accumulator, handed back sign-extended
// (dsp_runtime.c:769-794); the saturation stage (with the OUTPUT frame's dither) runs on it
__device__ __noinline__ int delayFirstFinish(int wv, int satKind, int satGainBits, int tv, int tpdfShift) {
    long long X = (long long)wv;
    if (satKind >= SAT_GAIN) { X >>= kMant; X = X * (long long)satGainBits; }
    if (satKind & 1) X += tpdfScaledI(tv, tpdfShift);
    return sat64_031_s32(X);
}

// post-ring word -> s.31 sample: fixed point stores it as such; the float class stores the (possibly not yet saturated)
// float and converts here (dspSaturateFloat0db + dsps31Float0DB, runtime/dsp_ieee754.h:60-83,170-184)
template <int CLS, bool FSMP = false> __device__ __forceinline__ int postToS31(int v) {
    if (CLS == ALU_F32) return FSMP ? __float_as_int(satF(__int_as_float(v))) : f2s31SatFast(v);      // DSP_FORMAT 5 stores the float itself
    return v;
}
// Phase B of the sink for interleaved output with NOUT (power of two) channels: 32/NOUT frames per pass.
template <int F, int NOUT, int CLS, bool FSMP>
__device__ __forceinline__ void storePassesT(int* __restrict__ out, unsigned rowA, unsigned p4, unsigned RM4, int mask,
                                             bool clean, int fw0, int fs, int T) {
    constexpr int FPP = 32 / NOUT, NPASS = F / FPP;
    if (clean) {
#pragma unroll
        for (int p = 0; p < NPASS; p++) out[p * 32] = postToS31<CLS, FSMP>(lds32(rowA + ((p4 + (unsigned)(p * FPP * 4)) & RM4))) & mask;
    } else {
#pragma unroll 1
        for (int p = 0; p < NPASS; p++) {
            const int ff = fw0 + p * FPP + fs;
            if (ff >= 0 && ff < T) out[p * 32] = postToS31<CLS, FSMP>(lds32(rowA + ((p4 + (unsigned)(p * FPP * 4)) & RM4))) & mask;
        }
    }
}
template <int F, int NOUT, int CLS>
__device__ __forceinline__ void storePasses(const bool fsmp, int* __restrict__ out, unsigned rowA, unsigned p4, unsigned RM4, int mask,
                                            bool clean, int fw0, int fs, int T) {
    if (CLS == ALU_F32 && fsmp) storePassesT<F, NOUT, CLS, true>(out, rowA, p4, RM4, mask, clean, fw0, fs, T);
    else storePassesT<F, NOUT, CLS, false>(out, rowA, p4, RM4, mask, clean, fw0, fs, T);
}

template <int K, int F, int CLS>
__global__ void __launch_bounds__(1024, 1)
k_chain2(const __grid_constant__ ChainPlan P, const Chain2Args A, const __grid_constant__ Chain2Geom G) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int NS = G.streamsPerCta, C = P.h.nChains, W = P.h.stateWords, T = A.nFrames;
    const int nSrc = P.h.nSrc;
    // helper warps take the LOW warp ids when G.helpersFirst (scheduler arbitration experiment)
    const int tid = G.helpersFirst ? (threadIdx.x < G.helpThreads ? threadIdx.x + G.secThreads : threadIdx.x - G.helpThreads) : threadIdx.x;
    const int lane = tid & 31;
    const int nStreamsRun = A.countPtr ? *A.countPtr : A.nStreams;      // exact second pass: as many streams as the pass before listed
    const int s0 = blockIdx.x * NS, nsHere = min(NS, nStreamsRun - s0);
    if (nsHere <= 0) return;
    const int* const smap = A.map;
    auto SX = [&](int local) -> int { return smap ? smap[s0 + local] : s0 + local; };      // position in the call's stream range
    const int nAll = G.secThreads + G.helpThreads;
    const int gmax = G.gmax;
    const int nTiles = (T + gmax + F - 1) / F;
    const int RM = G.postRing - 1;
    constexpr int XP = 2 * F + 1, AP = 2 * F + 1, TP = 4 * F + 1;        // row pitches (elements) of x / acc / tpdf rings

    if (CLS == ALU_F32 && tid < G.secThreads) {
        // =========================================================================== section warps, float ALU
        int* x_s = reinterpret_cast<int*>(smem_raw + G.xOff);
        int* post_s = reinterpret_cast<int*>(smem_raw + G.postOff);
        Lane2F<K> L;
        FltGuard mn;                       // exactness guard (avdsp_dev.cuh): smallest guard word of every value seen
        bool coefBad = false;              // a table coefficient outside what the guard can bound (fltCoefOutOfRange)
        const ChainLane e = A.lanes[tid];
        const bool live = e.slot >= 0 && e.slot / C < nsHere;
        const bool head = (e.flags & 1) != 0, tail = (e.flags & 2) != 0;
        const int g0 = e.firstSec;
        const int slot = e.slot < 0 ? 0 : e.slot;
        int* stLane = nullptr;
#pragma unroll
        for (int k = 0; k < K; k++) {
            L.acc[k] = L.x1[k] = L.x2[k] = L.y1[k] = L.y2[k] = 0.0f;
            L.b0[k] = L.b1[k] = L.b2[k] = L.a1[k] = L.a2[k] = 0.0f;
        }
        const ChainDesc& d = P.chains[slot % C];
        if (live) {
            stLane = A.state + (size_t)SX(slot / C) * W;
#pragma unroll
            for (int k = 0; k < K; k++) {
                const int sec = g0 + k;
                int cf[5];
                const bool tab = A.coefs && sec < d.nsec;
                sectionCoefs(P.pool + d.coefOff + 5 * sec, tab ? A.coefs : nullptr, A.coefPitch, tab ? P.pool[d.coefColOff + sec] : 0, SX(slot / C), cf);
                if (tab) for (int q = 0; q < 5; q++) coefBad |= fltCoefOutOfRange(cf[q]);
                L.b0[k] = __int_as_float(cf[0]); L.b1[k] = __int_as_float(cf[1]); L.b2[k] = __int_as_float(cf[2]);
                L.a1[k] = __int_as_float(cf[3]); L.a2[k] = __int_as_float(cf[4]);
                const int* q = stLane + P.pool[d.secStateOff + sec];        // [acc, -, x1, x2, y1, y2] (dsp_biquadSTD.h:84-119)
                L.acc[k] = __int_as_float(q[0]);
                L.x1[k] = __int_as_float(q[2]); L.x2[k] = __int_as_float(q[3]); L.y1[k] = __int_as_float(q[4]); L.y2[k] = __int_as_float(q[5]);
                fltGuard(mn, L.acc[k]); fltGuard(mn, L.x1[k]); fltGuard(mn, L.x2[k]); fltGuard(mn, L.y1[k]); fltGuard(mn, L.y2[k]);
            }
            if (coefBad) mn.mn = 0u;
        }
        const int* xrow = x_s + (size_t)((slot / C) * nSrc + max(d.srcId, 0)) * XP;
        int* prow = post_s + (size_t)slot * G.postPitch;
        for (int i = 0; i < nTiles; i++) {
            barSync(kBarFull + (i & 1), nAll);
            const int* xs = xrow + (i & 1) * F;
            const int t0 = i * F;
            int* ps = prow + (t0 & RM);
            if (A.exact) {
#pragma unroll 1
                for (int j = 0; j < F; j++) {
                    float x = __shfl_up_sync(0xffffffffu, L.y1[K - 1], 1);
                    if (head) x = __int_as_float(xs[j]);
                    laneStepPredF<K, true>(L, x, t0 + j, g0, T, mn);
                    if (tail && (unsigned)(t0 + j - g0 - (K - 1)) < (unsigned)T) ps[j] = __float_as_int(L.acc[K - 1]);
                }
            } else if (t0 >= gmax && t0 + F <= T) {
                if constexpr (K == 2) {
                    Lane2FP Q;
                    packLane(L, Q);
#pragma unroll 1
                    for (int j0 = 0; j0 < F; j0 += UNR) {
#pragma unroll
                        for (int jj = 0; jj < UNR; jj++) {
                            const int j = j0 + jj;
                            float x = __shfl_up_sync(0xffffffffu, hiF2(Q.y1), 1);
                            if (head) { x = __int_as_float(xs[j]); fltGuard(mn, x); }
                            if (jj % 6 == 0) laneStepFP<true>(Q, x, mn); else laneStepFP<false>(Q, x, mn);
                            if (tail) ps[j] = __float_as_int(hiF2(Q.acc));
                        }
                    }
                    unpackLane(Q, L);
                } else {
#pragma unroll 1
                for (int j0 = 0; j0 < F; j0 += UNR) {
#pragma unroll
                    for (int jj = 0; jj < UNR; jj++) {
                        const int j = j0 + jj;
                        float x = __shfl_up_sync(0xffffffffu, L.y1[K - 1], 1);
                        if (head) { x = __int_as_float(xs[j]); fltGuard(mn, x); }
                        if (jj % 6 == 0) laneStepF<K, true>(L, x, mn); else laneStepF<K, false>(L, x, mn);
                        if (tail) ps[j] = __float_as_int(L.acc[K - 1]);     // the sink saturates / converts (satF is idempotent)
                    }
                }
                }
            } else {
#pragma unroll 1
                for (int j = 0; j < F; j++) {
                    float x = __shfl_up_sync(0xffffffffu, L.y1[K - 1], 1);
                    if (head) { x = __int_as_float(xs[j]); if ((unsigned)(t0 + j - g0) < (unsigned)T) fltGuard(mn, x); }
                    laneStepPredF<K>(L, x, t0 + j, g0, T, mn);
                    if (tail && (unsigned)(t0 + j - g0 - (K - 1)) < (unsigned)T) ps[j] = __float_as_int(L.acc[K - 1]);
                }
            }
            barArrive(kBarDone + (i & 1), nAll);
        }
        if (live) {
#pragma unroll
            for (int k = 0; k < K; k++) {
                int* q = stLane + P.pool[d.secStateOff + g0 + k];
                q[0] = __float_as_int(L.acc[k]);
                q[2] = __float_as_int(L.x1[k]); q[3] = __float_as_int(L.x2[k]); q[4] = __float_as_int(L.y1[k]); q[5] = __float_as_int(L.y2[k]);
            }
            if (!A.exact && fltGuardFired(mn) && A.redo) A.redo[SX(slot / C)] = 1;
        }
        return;
    }
    if (CLS == ALU_INT64 && tid < G.secThreads) {
        // =========================================================================== section warps
        long long* acc_s = reinterpret_cast<long long*>(smem_raw);
        int* x_s = reinterpret_cast<int*>(smem_raw + G.xOff);
        int* post_s = reinterpret_cast<int*>(smem_raw + G.postOff);
        Lane2<K> L;
        const ChainLane e = A.lanes[tid];
        const bool live = e.slot >= 0 && e.slot / C < nsHere;
        const bool head = (e.flags & 1) != 0, tail = (e.flags & 2) != 0;
        const int g0 = e.firstSec;                       // frame lag of this lane's first section
        const int slot = e.slot < 0 ? 0 : e.slot;
        int* stLane = nullptr;
#pragma unroll
        for (int k = 0; k < K; k++) {
            L.acc[k] = 0; L.x1[k] = L.x2[k] = L.y1[k] = L.y2[k] = 0;
            L.b0[k] = L.b1[k] = L.b2[k] = L.a1[k] = L.a2[k] = 0;
        }
        const ChainDesc& d = P.chains[slot % C];
        if (live) {
            stLane = A.state + (size_t)SX(slot / C) * W;
#pragma unroll
            for (int k = 0; k < K; k++) {
                const int sec = g0 + k;
                int cf[5];
                const bool tab = A.coefs && sec < d.nsec;
                sectionCoefs(P.pool + d.coefOff + 5 * sec, tab ? A.coefs : nullptr, A.coefPitch, tab ? P.pool[d.coefColOff + sec] : 0, SX(slot / C), cf);
                L.b0[k] = cf[0]; L.b1[k] = cf[1]; L.b2[k] = cf[2]; L.a1[k] = cf[3]; L.a2[k] = cf[4];
                const int* q = stLane + P.pool[d.secStateOff + sec];
                L.acc[k] = (long long)(((unsigned long long)(unsigned)q[1] << 32) | (unsigned)q[0]);
                L.x1[k] = q[2]; L.x2[k] = q[3]; L.y1[k] = q[4]; L.y2[k] = q[5];
            }
        }
        const int* xrow = x_s + (size_t)((slot / C) * nSrc + max(d.srcId, 0)) * XP;
        long long* arow = acc_s + (size_t)((slot / C) * P.h.nAcc + max(d.accRow, 0)) * AP;
        int* prow = post_s + (size_t)slot * G.postPitch;
        const bool tail64 = tail && d.accRow >= 0;       // the sink needs the full accumulator (gain / dither ahead of the saturation)
        int* ck = reinterpret_cast<int*>(smem_raw + G.ckOff) + tid;       // [6K words][secThreads]: tile-start checkpoint of this lane
        const int CKP = G.secThreads;

        for (int i = 0; i < nTiles; i++) {
            barSync(kBarFull + (i & 1), nAll);
            const int* xs = xrow + (i & 1) * F;
            long long* as = arow + (i & 1) * F;
            const int t0 = i * F;
            int* ps = prow + (t0 & RM);
            if (t0 >= gmax && t0 + F <= T) {
                // checkpoint (shared memory: the LSU pipe is idle in this loop), optimistic tile, one test, rare replay
#pragma unroll
                for (int k = 0; k < K; k++) {
                    ck[(6 * k + 0) * CKP] = lo32(L.acc[k]); ck[(6 * k + 1) * CKP] = hi32(L.acc[k]);
                    ck[(6 * k + 2) * CKP] = L.x1[k]; ck[(6 * k + 3) * CKP] = L.x2[k];
                    ck[(6 * k + 4) * CKP] = L.y1[k]; ck[(6 * k + 5) * CKP] = L.y2[k];
                }
                unsigned worst = 0;
                // unrolled in groups of UNR steps (immediate offsets inside a group): the section loop stays a few KB of code
#pragma unroll 1
                for (int j0 = 0; j0 < F; j0 += UNR) {
#pragma unroll
                    for (int jj = 0; jj < UNR; jj++) {
                        const int j = j0 + jj;
                        int x = __shfl_up_sync(0xffffffffu, L.y1[K - 1], 1);
                        if (head) x = xs[j];
                        laneStepFast<K>(L, x, worst);
                        if (tail) ps[j] = L.y1[K - 1];
                        if (tail64) as[j] = L.acc[K - 1];
                    }
                }
                if (__any_sync(0xffffffffu, worst > kSatLimit)) {
                    // some section of this warp saturated somewhere in the tile: replay it exactly
#pragma unroll
                    for (int k = 0; k < K; k++) {
                        L.acc[k] = (long long)(((unsigned long long)(unsigned)ck[(6 * k + 1) * CKP] << 32) | (unsigned)ck[(6 * k + 0) * CKP]);
                        L.x1[k] = ck[(6 * k + 2) * CKP]; L.x2[k] = ck[(6 * k + 3) * CKP];
                        L.y1[k] = ck[(6 * k + 4) * CKP]; L.y2[k] = ck[(6 * k + 5) * CKP];
                    }
#pragma unroll 1
                    for (int j = 0; j < F; j++) {
                        int x = __shfl_up_sync(0xffffffffu, L.y1[K - 1], 1);
                        if (head) x = xs[j];
                        laneStepExact<K>(L, x);
                        if (tail) ps[j] = L.y1[K - 1];
                        if (tail64) as[j] = L.acc[K - 1];
                    }
                }
            } else {
#pragma unroll 1
                for (int j = 0; j < F; j++) {
                    int x = __shfl_up_sync(0xffffffffu, L.y1[K - 1], 1);
                    if (head) x = xs[j];
                    laneStepPred<K>(L, x, t0 + j, g0, T);
                    if (tail && (unsigned)(t0 + j - g0 - (K - 1)) < (unsigned)T) ps[j] = L.y1[K - 1];
                    if (tail64) as[j] = L.acc[K - 1];
                }
            }
            barArrive(kBarDone + (i & 1), nAll);
        }
        if (live) {
#pragma unroll
            for (int k = 0; k < K; k++) {
                int* q = stLane + P.pool[d.secStateOff + g0 + k];
                q[0] = (int)L.acc[k]; q[1] = (int)(L.acc[k] >> 32);
                q[2] = L.x1[k]; q[3] = L.x2[k]; q[4] = L.y1[k]; q[5] = L.y2[k];
            }
        }
        return;
    }

    // =============================================================================== helper warps
    const int ht = tid - G.secThreads, hw = ht >> 5, nHW = G.helpThreads >> 5;
    const bool fsmp = CLS == ALU_F32 && !P.h.sampleInt;       // DSP_FORMAT 5: float samples in, floats out, no STORE mask
    const int storeMask = fsmp ? -1 : ditherMask(P.h.storeDither);
    const bool hasCalc = P.h.hasTpdfCalc != 0;
    const unsigned sb = smemAddr(smem_raw);
    int* post_s = reinterpret_cast<int*>(smem_raw + G.postOff);
    int* tpdf_s = reinterpret_cast<int*>(smem_raw + G.tpdfOff);
    int* ridx_s = reinterpret_cast<int*>(smem_raw + G.ridxOff);            // [slots] effective delay-ring index at launch start
    int* stale_s = ridx_s + NS * C;                                        // [slots] stale ring index (>= n) or -1
    int* sfix_s = stale_s + NS * C;                                        // [slots] stale case: ring[n-1], restored over post(0)
    // warp 0 doubles as the dither PRNG: lane = stream
    Prng g = {0, 0, 0, 0}; int tpdfValue = 0, tpdfRandom = 0, dith = 0; bool drew = false;
    int* auxp = nullptr;
    if (hw == 0 && lane < nsHere) {
        auxp = A.state + (size_t)SX(lane) * W + P.h.auxOff;
        g.s0 = auxp[AUX_S0]; g.s1 = auxp[AUX_S1]; g.s2 = auxp[AUX_S2]; g.s3 = auxp[AUX_S3];
        tpdfValue = auxp[AUX_TPDF_VALUE]; tpdfRandom = auxp[AUX_TPDF_RANDOM]; dith = auxp[AUX_DITHER];
    }
    // Stream ownership: every helper warp but the PRNG warp owns the streams sl = ow, ow+nOwn, ... for the
    // whole launch (their post rings and delay state are warp-private: only __syncwarp inside the sink).
    const bool prngOnly = hasCalc && nHW > 1 && hw == 0;
    const int ow = (hasCalc && nHW > 1) ? hw - 1 : hw;
    const int nOwn = (hasCalc && nHW > 1) ? nHW - 1 : nHW;
    const bool vecOut = A.outChStride == 1 && (P.h.nOut & 3) == 0 && (A.outFrameStride & 3) == 0 &&
                        (A.outStreamStride & 3) == 0 && ((size_t)A.out & 15) == 0;

    // ---- delay lines.  Reference semantics (dsp_runtime.c:769-794): ring of n samples, frame f swaps with
    // position (idx0+f) mod n, so the output of frame f is the post value of frame f-n.  Here the post ring
    // (R >= 2F + gmax + n steps of history) IS the delay line: the prologue preloads the n samples the
    // reference ring holds as "virtual frames" -n..-1, the epilogue writes the last n back in ring layout.
    // A stale index idx0 >= n (delay shortened by reload_params) is used once by the reference and then
    // wraps to 0: frame 0 swaps with ring[idx0], frames >= 1 behave like idx0 = n-1.
    bool anyStale = false;
    if (!prngOnly)
        for (int sl = ow; sl < nsHere; sl += nOwn) {
            int* st = A.state + (size_t)SX(sl) * W;
            for (int c = 0; c < C; c++) {
                const ChainDesc& d = P.chains[c];
                const int n = d.delayN;
                if (n <= 0) continue;
                const int gc = d.nsec > 0 ? d.nsec - 1 : 0;
                const int* ring = st + d.delayOff + 1;
                const int idx0 = st[d.delayOff];
                const bool stale = idx0 >= n || idx0 < 0;
                anyStale |= stale;
                int* prow = post_s + (size_t)(sl * C + c) * G.postPitch;
                for (int k = lane; k < n; k += 32) {          // virtual frame j = k - n feeds output frame k
                    int v;
                    if (!stale) v = ring[(idx0 + k) % n];
                    else v = (k == 0) ? ring[idx0] : ring[k - 1];
                    prow[(k - n + gc) & RM] = v;
                }
                if (lane == 0) {
                    ridx_s[sl * C + c] = stale ? n - 1 : idx0; stale_s[sl * C + c] = stale ? idx0 : -1;
                    if (stale) { sfix_s[sl * C + c] = ring[n - 1]; prow[gc & RM] = ring[n - 1]; }   // takes the place of post(0), see above
                }
            }
        }
    __syncwarp();

    // ---- input PCM tiles by TMA: lane 0 of every owner warp issues, two tiles ahead, one bulk copy per owned
    // stream (interleaved: F*nIn contiguous words) or per (stream, channel) (planar: F contiguous words) into
    // the raw tiles; completion is counted in bytes on the warp's mbarrier of that parity.  Tiles that cannot go
    // through TMA (partial last tile, misaligned caller buffers) are read with plain loads instead.
    const int nIn = P.h.nIn;
    const int rowBytes = F * nIn * 4;
    const bool interleavedIn = A.inChStride == 1 && A.inFrameStride == nIn;
    const bool planarIn = A.inFrameStride == 1;
    const bool tmaOk = G.rawOff != 0 && nSrc > 0 && nIn > 0 && ((size_t)A.in & 15) == 0 && (A.inStreamStride & 3) == 0 &&
                       ((interleavedIn && (rowBytes & 15) == 0) || (planarIn && !interleavedIn && (A.inChStride & 3) == 0 && (F & 3) == 0));
    const unsigned rawFB = interleavedIn ? nIn * 4 : 4, rawCB = interleavedIn ? 4 : F * 4;   // frame / channel stride (bytes) in a staged tile
    const unsigned mbar0 = sb + G.mbarOff + 16 * hw;
    if (tmaOk && !prngOnly && lane == 0) { mbarInit(mbar0, 1); mbarInit(mbar0 + 8, 1); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
    __syncwarp();
    auto tileUsesTma = [&](int it) { return tmaOk && (it + 1) * F <= T; };
    auto issueTile = [&](int it) {
        if (prngOnly || !tileUsesTma(it)) return;
        __syncwarp();                                    // every lane is done reading the buffer being refilled
        fenceProxyAsync();
        const unsigned bar = mbar0 + 8 * (it & 1);
        const int cnt = nsHere > ow ? (nsHere - ow + nOwn - 1) / nOwn : 0;      // streams this warp owns
        // lane 0 posts the byte count (the phase cannot complete before this arrival, so the order against the copies
        // below does not matter); lane j issues the copy of the warp's j-th stream -- in parallel, not in a lane-0 loop
        if (lane == 0) mbarExpectTx(bar, (unsigned)(cnt * rowBytes));
        for (int j = lane; j < cnt; j += 32) {
            const int sl = ow + j * nOwn;
            const int* src = A.in + (size_t)SX(sl) * A.inStreamStride + (size_t)(it * F) * A.inFrameStride;
            const unsigned dst = sb + G.rawOff + sl * G.rawStreamBytes + (it & 1) * rowBytes;
            if (interleavedIn) tmaLoad1D(dst, src, (unsigned)rowBytes, bar);
            else for (int ch = 0; ch < nIn; ch++) tmaLoad1D(dst + ch * F * 4, src + (size_t)ch * A.inChStride, (unsigned)(F * 4), bar);
        }
    };

    bool simpleSrc = !fsmp;                                 // every source is LOAD_GAIN of a fed input (int32 samples)
    for (int k = 0; k < nSrc && k < kFastTab; k++) simpleSrc = simpleSrc && P.h.sKind[k] == SRC_LOAD_GAIN && P.h.sCh[k] >= 0;
    // ---- source stage of tile `it`: frames [it*F, it*F+F) -> x ring (one value per distinct source), dither values
    auto sourceTile = [&](int it) {
        const int f0 = it * F;
        if (f0 >= T) return;
        if (G.debugSkip & 1) { issueTile(it + 2); return; }
        if (hw == 0 && lane < nsHere && !(G.debugSkip & 2)) {
            int* row = tpdf_s + lane * TP + (it & 3) * F;
            const int n = min(F, T - f0);
            if (hasCalc) {
                for (int j = 0; j < n; j++) {
                    if (dith == P.h.tpdfDither) { tpdfValue = tpdfDraw(g, tpdfRandom); drew = true; }
                    else dith = P.h.tpdfDither;      // table switch on the first frame after a reset: no draw (dsp_runtime.c:539-544)
                    row[j] = tpdfValue;
                }
            } else {
                for (int j = 0; j < n; j++) row[j] = tpdfValue;
            }
        }
        if (nSrc == 0 || prngOnly) return;
        const bool staged = tileUsesTma(it);
        if (staged) mbarWait(mbar0 + 8 * (it & 1), (unsigned)((it >> 1) & 1));
        if (simpleSrc && staged && lane < F && f0 + lane < T) {
            // the common source stage (fixed point, every source LOAD_GAIN of a fed input, tile staged by TMA) as its own
            // compact loop, apart from the general forms below
            unsigned xa = sb + G.xOff + ow * G.xStreamBytes + ((it & 1) * F + lane) * 4;
            unsigned ra = sb + G.rawOff + ow * G.rawStreamBytes + (it & 1) * rowBytes + lane * rawFB;
            for (int sl = ow; sl < nsHere; sl += nOwn, xa += nOwn * G.xStreamBytes, ra += nOwn * G.rawStreamBytes) {
#pragma unroll
                for (int k = 0; k < kFastTab; k++) {
                    if (k >= nSrc) break;
                    const int smp = lds32(ra + (interleavedIn ? (unsigned)(P.h.sCh[k] * 4) : (unsigned)(P.h.sCh[k] * F * 4)));
                    if (CLS == ALU_F32) {
                        // LOAD_GAIN in the float class: hardware convert + mul.rz.ftz when the host checked that no product
                        // can reach the underflow range (G.floatFast: every gain in [2^-30, 2^30]), else the restatement
                        float xf = G.floatFast ? mulFF_fast(i2f31Fast(smp), __int_as_float(P.h.sArg[k]))
                                               : mulFF(i2fScaled(smp, 31), __int_as_float(P.h.sArg[k]));
                        if (smp == 0) xf = 0.0f;                       // the reference's product of a zero is +0, never -0
                        sts32(xa + G.srcXOff[k], __float_as_int(xf));
                    } else sts32(xa + G.srcXOff[k], q59ToS31(mul32(smp, P.h.sArg[k])));
                }
            }
        } else if (lane < F && f0 + lane < T) {
            unsigned xa = sb + G.xOff + ow * G.xStreamBytes + ((it & 1) * F + lane) * 4;
            unsigned ra = sb + G.rawOff + ow * G.rawStreamBytes + (it & 1) * rowBytes + lane * rawFB;
            for (int sl = ow; sl < nsHere; sl += nOwn, xa += nOwn * G.xStreamBytes, ra += nOwn * G.rawStreamBytes) {
                const int* in = A.in + (size_t)SX(sl) * A.inStreamStride + (size_t)(f0 + lane) * A.inFrameStride;
                if (simpleSrc && staged) {
                    // common case, branch-free: LOAD_GAIN sources read from the TMA-staged tile
#pragma unroll
                    for (int k = 0; k < kFastTab; k++) {
                        if (k >= nSrc) break;
                        const int smp = lds32(ra + (interleavedIn ? (unsigned)(P.h.sCh[k] * 4) : (unsigned)(P.h.sCh[k] * F * 4)));
                        if (CLS == ALU_F32) {
                            // LOAD_GAIN in the float class: hardware convert + mul.rz.ftz when the host checked that no product
                            // can reach the underflow range (G.floatFast: every gain in [2^-30, 2^30]), else the restatement
                            float xf = G.floatFast ? mulFF_fast(i2f31Fast(smp), __int_as_float(P.h.sArg[k]))
                                                   : mulFF(i2fScaled(smp, 31), __int_as_float(P.h.sArg[k]));
                            if (smp == 0) xf = 0.0f;                   // the reference's product of a zero is +0, never -0
                            sts32(xa + G.srcXOff[k], __float_as_int(xf));
                        }
                        else sts32(xa + G.srcXOff[k], q59ToS31(mul32(smp, P.h.sArg[k])));
                    }
                    continue;
                }
                if (CLS == ALU_F32) {            // float class, any source kind: straight from global memory
                    for (int k = 0; k < nSrc; k++)
                        sts32(xa + (unsigned)(k * XP * 4), __float_as_int(chainSourceF(P, P.chains[P.h.srcChain[k]], in, A.inChStride)));
                    continue;
                }
                // flattened source tables with static indices: constant-bank operands, no descriptor loads
#pragma unroll
                for (int k = 0; k < kFastTab; k++) {
                    if (k >= nSrc) break;                    // early exit: no chain of skipped-iteration tests
                    {
                        long long X;
                        if (P.h.sKind[k] == SRC_LOAD_MUX) {
                            const ChainDesc& d = P.chains[P.h.srcChain[k]];
                            X = staged ? muxFromShared(P, d, ra, rawCB) : chainSource(P, d, in, A.inChStride);
                        } else {
                            int smp = 0;
                            if (P.h.sCh[k] >= 0) smp = staged ? lds32(ra + P.h.sCh[k] * rawCB) : in[(size_t)P.h.sCh[k] * A.inChStride];
                            X = (P.h.sKind[k] == SRC_LOAD_GAIN) ? mul32(smp, P.h.sArg[k]) : (long long)smp;
                        }
                        sts32(xa + G.srcXOff[k], q59ToS31(X));
                    }
                }
            }
        }
        issueTile(it + 2);                               // refill this parity's buffer two tiles ahead
    };

    bool simpleA = CLS == ALU_INT64 && !anyStale && !(G.debugSkip & 8);             // all post-processed chains are cascade -> SAT0DB_TPDF
    for (int k = 0; k < P.h.nProc && k < kFastTab; k++) simpleA = simpleA && P.h.pFlags[k] == (PF_SECTIONS | PF_SAT_TPDF);
    const bool tpdfUp = P.h.tpdfShift >= 0;                    // warp-uniform: the dither is shifted up (usual) or down
    const int tpdfSh = (tpdfUp ? P.h.tpdfShift : -P.h.tpdfShift) & 63;
    // ---- per-lane constants of the (frame-in-pass, channel) store mapping (interleaved output, F == 32)
    const int nOut = P.h.nOut;
    const bool laneOut = F == 32 && A.outChStride == 1 && A.outFrameStride == nOut && nOut <= 16 && (nOut & (nOut - 1)) == 0 &&
                         P.h.nDelayFirst == 0;            // delay-first paths are finished by the frame-per-lane form of stage B
    const int fpp = laneOut ? 32 / nOut : 1;                  // frames per pass
    const int bCh = lane % nOut, bFs = lane / nOut;
    const int bChain = P.h.chainOfOut[bCh];
    const unsigned bRow = bChain >= 0 ? (unsigned)(bChain * G.postPitch * 4) : 0u;
    const unsigned bPos4 = (unsigned)((bFs + P.h.outOff[bCh]) * 4);
    // outputs no path writes read as 0; DSP_LOAD_STORE copies are not masked by the STORE dither mask
    const int bMask = bChain >= 0 ? (P.chains[bChain].srcKind == SRC_RAW ? -1 : storeMask) : 0;

    auto isProc = [&](int c) { for (int k = 0; k < P.h.nProc; k++) if (P.h.procChain[k] == c) return true; return false; };
    // ---- sink stage of window `iw`
    auto sinkWindow = [&](int iw) {
        if (prngOnly || lane >= F || (G.debugSkip & 4)) return;
        const unsigned wmask = F == 32 ? 0xffffffffu : ((1u << (F & 31)) - 1u);
        const int t = iw * F + lane;
        const unsigned tpos4 = (unsigned)(t & RM) << 2, RM4 = (unsigned)RM << 2;
        const int f = iw * F - gmax + lane;                  // the output frame this lane stores in phase B
        const unsigned f4 = (unsigned)f << 2;
        unsigned postA = sb + G.postOff + ow * G.postStreamBytes;
        unsigned accA = sb + ow * G.accStreamBytes + ((iw & 1) * F + lane) * 8;
        unsigned tpdfA = sb + G.tpdfOff + ow * G.tpdfStreamBytes;
        if (((CLS == ALU_INT64 && simpleA) || (CLS == ALU_F32 && P.h.nProc == 0)) && laneOut && !anyStale && iw * F >= gmax && (iw + 1) * F <= T &&
            !(G.debugSkip & 16)) {
            // the common window of the common program (every post-processed chain is cascade -> SAT0DB_TPDF, interleaved
            // power-of-two outputs, interior tile, no stale ring index) as its own compact loop: nothing of the general
            // forms below sits between its instructions (the kernel is instruction-cache sensitive)
            const int fw0 = iw * F - gmax;
            const unsigned p4 = (unsigned)(fw0 << 2) + bPos4;
            for (int sl = ow; sl < nsHere; sl += nOwn, postA += nOwn * G.postStreamBytes, accA += nOwn * G.accStreamBytes, tpdfA += nOwn * G.tpdfStreamBytes) {
                if (CLS == ALU_INT64) {
#pragma unroll
                    for (int k = 0; k < kFastTab; k++) {
                        if (k >= P.h.nProc) break;
                        long long X = lds64(accA + G.pAccOff[k]);
                        const long long tv = lds32(tpdfA + ((unsigned)((t - P.h.pLag[k]) & (4 * F - 1)) << 2));
                        X += tpdfUp ? (long long)((unsigned long long)tv << tpdfSh) : (tv >> tpdfSh);
                        sts32(postA + G.pPostOff[k] + tpos4, sat64_031_s32(X));
                    }
                    __syncwarp(wmask);
                }
                int* out = A.out + (size_t)SX(sl) * A.outStreamStride + (size_t)fw0 * A.outFrameStride + lane;
                const unsigned rowA = postA + bRow;
                switch (nOut) {
                case 1:  storePasses<F, 1, CLS>(fsmp, out, rowA, p4, RM4, bMask, true, fw0, bFs, T); break;
                case 2:  storePasses<F, 2, CLS>(fsmp, out, rowA, p4, RM4, bMask, true, fw0, bFs, T); break;
                case 4:  storePasses<F, 4, CLS>(fsmp, out, rowA, p4, RM4, bMask, true, fw0, bFs, T); break;
                case 8:  storePasses<F, 8, CLS>(fsmp, out, rowA, p4, RM4, bMask, true, fw0, bFs, T); break;
                default: storePasses<F, 16, CLS>(fsmp, out, rowA, p4, RM4, bMask, true, fw0, bFs, T); break;
                }
                __syncwarp(wmask);
            }
            return;
        }
        for (int sl = ow; sl < nsHere; sl += nOwn, postA += nOwn * G.postStreamBytes, accA += nOwn * G.accStreamBytes, tpdfA += nOwn * G.tpdfStreamBytes) {
            // A: step t of every chain that needs post-processing: accumulator (or inline source) -> [gain] -> saturate
            //    (+dither, +gain) -> post ring (dsp_runtime.c:464-534, 636-640).  Direct chains were written by their tails.
            if (CLS == ALU_F32) {
                // float class: the tail lanes left the cascade's accumulator (float bits) in the post ring; chains with
                // gain / dither are finished in place, the others are saturated and converted by stage B
                for (int k = 0; k < P.h.nProc; k++) {
                    const int c = P.h.procChain[k];
                    const ChainDesc& d = P.chains[c];
                    const int fk = t - (d.nsec > 0 ? d.nsec - 1 : 0);
                    if (fk < 0 || fk >= T) continue;
                    const unsigned pa = postA + (unsigned)(c * G.postPitch * 4) + tpos4;
                    float X;
                    if (d.nsec > 0) X = __int_as_float(lds32(pa));
                    else {
                        X = chainSourceF(P, d, A.in + (size_t)SX(sl) * A.inStreamStride + (size_t)fk * A.inFrameStride, A.inChStride);
                        if (d.srcKind == SRC_LOAD_MUX && fk == T - 1) A.state[(size_t)SX(sl) * W + d.muxStateOff] = __float_as_int(X);
                    }
                    const int flags = (d.hasGain ? PF_GAIN : 0) | ((d.satKind & 1) ? PF_SAT_TPDF : 0) | (d.satKind >= SAT_GAIN ? PF_SAT_GAIN : 0);
                    const int tv = (flags & PF_SAT_TPDF) ? lds32(tpdfA + ((unsigned)(fk & (4 * F - 1)) << 2)) : 0;
                    const int v = __float_as_int(finishF(X, flags, d.gainBits, d.satGainBits, tv, P.h.storeDither));
                    if (anyStale && fk == 0 && d.delayN > 0 && stale_s[sl * C + c] >= 0)
                        A.state[(size_t)SX(sl) * W + d.delayOff + 1 + stale_s[sl * C + c]] = v;
                    else sts32(pa, v);
                }
            } else if (simpleA && iw * F >= gmax && (iw + 1) * F <= T) {
                // common case, branch-free: every post-processed chain is cascade -> SAT0DB_TPDF and the window is interior
#pragma unroll
                for (int k = 0; k < kFastTab; k++) {
                    if (k >= P.h.nProc) break;
                    long long X = lds64(accA + G.pAccOff[k]);
                    const long long tv = lds32(tpdfA + ((unsigned)((t - P.h.pLag[k]) & (4 * F - 1)) << 2));
                    X += tpdfUp ? (long long)((unsigned long long)tv << tpdfSh) : (tv >> tpdfSh);
                    sts32(postA + G.pPostOff[k] + tpos4, sat64_031_s32(X));
                }
            } else
#pragma unroll
            for (int k = 0; k < kFastTab; k++) {
                if (k >= P.h.nProc || (G.debugSkip & 8)) break;
                {
                    const int fk = t - P.h.pLag[k];
                    if (fk >= 0 && fk < T) {
                        const int flags = P.h.pFlags[k];
                        long long X;
                        if (flags & PF_SECTIONS) X = lds64(accA + G.pAccOff[k]);
                        else {
                            const ChainDesc& d = P.chains[P.h.pChain[k]];
                            X = chainSource(P, d, A.in + (size_t)SX(sl) * A.inStreamStride + (size_t)fk * A.inFrameStride, A.inChStride);
                            if (d.srcKind == SRC_LOAD_MUX && fk == T - 1) {
                                int* st = A.state + (size_t)SX(sl) * W;
                                st[d.muxStateOff] = lo32(X); st[d.muxStateOff + 1] = hi32(X);
                            }
                        }
                        if (flags & PF_GAIN) X = X * (long long)P.h.pGain[k];
                        if (flags & PF_SAT_GAIN) { X >>= kMant; X = X * (long long)P.h.pSatGain[k]; }
                        if (flags & PF_SAT_TPDF) {
                            const long long tv = lds32(tpdfA + ((unsigned)(fk & (4 * F - 1)) << 2));
                            X += tpdfUp ? (long long)((unsigned long long)tv << tpdfSh) : (tv >> tpdfSh);      // dspTpdfApply, dsp_tpdf.h:141-145
                        }
                        // LOAD_STORE: the sample itself; delay-first paths: the accumulator's low word (what the ring stores)
                        const int v = (flags & (PF_RAW | PF_DELAY_FIRST)) ? lo32(X) : sat64_031_s32(X);
                        if (anyStale && fk == 0 && P.h.pDelayN[k] > 0 && stale_s[sl * C + P.h.pChain[k]] >= 0)
                            A.state[(size_t)SX(sl) * W + P.chains[P.h.pChain[k]].delayOff + 1 + stale_s[sl * C + P.h.pChain[k]]] = v;
                        else sts32(postA + G.pPostOff[k] + tpos4, v);
                    }
                }
            }
            // stale delay index on a cascade (rare): the tail lane stored a value where the preloaded ring[n-1] has to stay
            if (anyStale && iw * F <= gmax && lane == 0)
                for (int c = 0; c < C; c++) {
                    const ChainDesc& d = P.chains[c];
                    if (d.nsec > 0 && d.delayN > 0 && stale_s[sl * C + c] >= 0 && (d.nsec - 1) / F == iw) {
                        // every tail lane stores its y1 at the slot of frame 0; a direct chain's is the real post(0)
                        // (a post-processed chain's post(0) was sent to ring[idx0] by stage A above)
                        int* pr = post_s + (size_t)(sl * C + c) * G.postPitch + ((d.nsec - 1) & RM);
                        if (d.accRow < 0 && !(CLS == ALU_F32 && isProc(c)))
                            A.state[(size_t)SX(sl) * W + d.delayOff + 1 + stale_s[sl * C + c]] = CLS == ALU_F32 ? __float_as_int(satF(__int_as_float(*pr))) : *pr;
                        *pr = sfix_s[sl * C + c];
                    }
                }
            __syncwarp(wmask);
            // B: delayed read from the post ring + mask + store.
            if (G.debugSkip & 16) {
            } else if (laneOut) {
                // interleaved output, power-of-two channel count: lane = (frame inside a pass, channel); the 32 lanes of a
                // pass store one contiguous 128-byte run.  Per-lane constants (row, lag-delay) sit in registers and the
                // pass geometry is a template constant: a pass is add / and / add / LDS / and / STG with immediate offsets.
                const int fw0 = iw * F - gmax;
                int* out = A.out + (size_t)SX(sl) * A.outStreamStride + (size_t)fw0 * A.outFrameStride + lane;
                const unsigned rowA = postA + bRow;
                const unsigned p4 = (unsigned)(fw0 << 2) + bPos4;           // 4*(post-ring step of this lane's element in pass 0)
                const bool clean = fw0 >= 0 && fw0 + F <= T;
                switch (nOut) {
                case 1:  storePasses<F, 1, CLS>(fsmp, out, rowA, p4, RM4, bMask, clean, fw0, bFs, T); break;
                case 2:  storePasses<F, 2, CLS>(fsmp, out, rowA, p4, RM4, bMask, clean, fw0, bFs, T); break;
                case 4:  storePasses<F, 4, CLS>(fsmp, out, rowA, p4, RM4, bMask, clean, fw0, bFs, T); break;
                case 8:  storePasses<F, 8, CLS>(fsmp, out, rowA, p4, RM4, bMask, clean, fw0, bFs, T); break;
                default: storePasses<F, 16, CLS>(fsmp, out, rowA, p4, RM4, bMask, clean, fw0, bFs, T); break;
                }
            } else if (f >= 0 && f < T) {
                // any layout: lane = frame, 16-byte stores when the layout allows
                int* out = A.out + (size_t)SX(sl) * A.outStreamStride + (size_t)f * A.outFrameStride;
#pragma unroll
                for (int ch0 = 0; ch0 < kFastTab; ch0 += 4) {
                    if (ch0 >= P.h.nOut) break;
                    int val[4];
#pragma unroll
                    for (int q = 0; q < 4; q++) {
                        const int ch = ch0 + q;
                        int v = 0;      // outputs no path writes read as 0 (io[] is zeroed at the start of every frame)
                        if (ch < P.h.nOut && P.h.chainOfOut[ch] >= 0) {
                            const ChainDesc& dc = P.chains[P.h.chainOfOut[ch]];
                            int wv = lds32(postA + G.outRowOff[ch] + ((f4 + (unsigned)G.outPos4[ch]) & RM4));
                            if (dc.delayFirst)      // out of line: rare program shape, keeps the common store loop compact
                                wv = delayFirstFinish(wv, dc.satKind, dc.satGainBits, lds32(tpdfA + ((unsigned)(f & (4 * F - 1)) << 2)), P.h.tpdfShift);
                            else wv = fsmp ? postToS31<CLS, true>(wv) : postToS31<CLS, false>(wv);      // float class: the ring holds the float (storePasses converts in the fast path)
                            v = wv & (dc.srcKind == SRC_RAW ? -1 : storeMask);
                        }
                        val[q] = v;
                    }
                    if (vecOut) *reinterpret_cast<int4*>(out + ch0) = make_int4(val[0], val[1], val[2], val[3]);
                    else {
#pragma unroll
                        for (int q = 0; q < 4; q++) if (ch0 + q < P.h.nOut) out[(size_t)(ch0 + q) * A.outChStride] = val[q];
                    }
                }
            }
            __syncwarp(wmask);
        }
    };

    issueTile(0);
    issueTile(1);
    sourceTile(0);
    barArrive(kBarFull + 0, nAll);
    for (int i = 0; i < nTiles; i++) {
        if (i + 1 < nTiles) { sourceTile(i + 1); barArrive(kBarFull + ((i + 1) & 1), nAll); }
        barSync(kBarDone + (i & 1), nAll);
        sinkWindow(i);
    }

    if (auxp) {
        auxp[AUX_S0] = g.s0; auxp[AUX_S1] = g.s1; auxp[AUX_S2] = g.s2; auxp[AUX_S3] = g.s3;
        auxp[AUX_TPDF_VALUE] = tpdfValue; auxp[AUX_TPDF_RANDOM] = tpdfRandom; auxp[AUX_DITHER] = dith;
        if (drew) {   // TPDF_CALC leaves its last value (as an ALU word) in the data area (dsp_runtime.c:541-543)
            int* q = A.state + (size_t)SX(lane) * W + P.h.tpdfDataOff;
            if (CLS == ALU_F32) q[0] = __float_as_int(i2fScaled(tpdfValue, 31));
            else { q[0] = tpdfValue; q[1] = tpdfValue >> 31; }
        }
    }
    if (prngOnly || T <= 0) return;
    __syncwarp();
    for (int sl = ow; sl < nsHere; sl += nOwn) {
        int* st = A.state + (size_t)SX(sl) * W;
        for (int c = 0; c < C; c++) {
            const ChainDesc& d = P.chains[c];
            // last LOAD_MUX value of chains with sections stays in the data area (dsp_runtime.c:893-896)
            if (d.srcKind == SRC_LOAD_MUX && d.nsec > 0 && lane == 0) {
                const int* fr = A.in + (size_t)SX(sl) * A.inStreamStride + (size_t)(T - 1) * A.inFrameStride;
                if (CLS == ALU_F32) st[d.muxStateOff] = __float_as_int(chainSourceF(P, d, fr, A.inChStride));
                else { const long long X = chainSource(P, d, fr, A.inChStride); st[d.muxStateOff] = (int)X; st[d.muxStateOff + 1] = (int)(X >> 32); }
            }
            // delay line back to the reference's ring layout: frame j sits at position (idx0+j) mod n
            const int n = d.delayN;
            if (n <= 0) continue;
            const int gc = d.nsec > 0 ? d.nsec - 1 : 0;
            const int idx0 = ridx_s[sl * C + c];
            const int* prow = post_s + (size_t)(sl * C + c) * G.postPitch;
            int* ring = st + d.delayOff + 1;
            for (int k = lane; k < n; k += 32) {
                const int j = T - n + k;                                     // frames T-n .. T-1 (virtual ones included)
                const int pv = prow[(j + gc) & RM];       // float class: direct chains still hold the unsaturated accumulator
                ring[(int)(((long long)idx0 + j + n) % n)] = CLS == ALU_F32 ? __float_as_int(satF(__int_as_float(pv))) : pv;
            }
            if (lane == 0) st[d.delayOff] = (int)(((long long)idx0 + T) % n);
        }
    }
}

// ------------------------------------------------------------------------------------------------
static int envInt2(const char* name, int dflt) { const char* v = getenv(name); return (v && *v) ? atoi(v) : dflt; }

// pack the section lanes of NS streams into warps (first-fit decreasing): a cascade never straddles a warp
static int packLanes2(const ChainPlan& p, int NS, int K, ChainLane* out, int* gmax) {
    struct Item { int slot, lanes; };
    std::vector<Item> items;
    const int C = p.h.nChains;
    int gm = 0;
    for (int s = 0; s < NS; s++)
        for (int c = 0; c < C; c++) {
            const int n = p.chains[c].nsec / K;
            if (n > 0) items.push_back({s * C + c, n});
            if (p.chains[c].nsec > 0) gm = std::max(gm, p.chains[c].nsec - 1);
        }
    if (gmax) *gmax = gm;
    std::stable_sort(items.begin(), items.end(), [](const Item& a, const Item& b) { return a.lanes > b.lanes; });
    std::vector<int> fill;
    std::vector<std::vector<Item>> warps;
    for (const Item& it : items) {
        if (it.lanes > 32) return -1;
        size_t w = 0;
        for (; w < fill.size(); w++) if (fill[w] + it.lanes <= 32) break;
        if (w == fill.size()) { fill.push_back(0); warps.emplace_back(); }
        fill[w] += it.lanes; warps[w].push_back(it);
    }
    const int threads = (int)fill.size() * 32;
    if (threads > 1024) return -1;
    if (out) {
        for (int i = 0; i < threads; i++) { out[i].slot = -1; out[i].depth = 0; out[i].flags = 0; out[i].firstSec = 0; }
        for (size_t w = 0; w < warps.size(); w++) {
            int l = (int)w * 32;
            for (const Item& it : warps[w])
                for (int dpt = 0; dpt < it.lanes; dpt++, l++) {
                    out[l].slot = it.slot; out[l].depth = dpt; out[l].firstSec = dpt * K;
                    out[l].flags = (dpt == 0 ? 1 : 0) | (dpt == it.lanes - 1 ? 2 : 0);
                }
        }
    }
    return threads;
}

// float class: the exactness guard of the cascades (avdsp_dev.cuh, fltGuard) bounds products through their operands, which needs
// every non-zero biquad coefficient within [2^-60, 2^7) (avdsp_dev.cuh, fltGuard; denormal coefficients are out)
bool chainFloatCoefsInRange(const ChainPlan& plan) {
    for (int c = 0; c < plan.h.nChains; c++) {
        const ChainDesc& d = plan.chains[c];
        for (int k = 0; k < 5 * d.nsec; k++) {
            const uint32_t u = (uint32_t)plan.pool[d.coefOff + k] & 0x7FFFFFFFu;
            const int ex = (int)(u >> 23);
            if (u != 0 && (ex < 127 - 60 || ex > 127 + 6)) return false;
        }
    }
    return true;
}

bool chain2Supports(const ChainPlan& plan) {
    if (plan.h.aluClass == ALU_F32 && !chainFloatCoefsInRange(plan)) return false;
    // the helper warps address everything through the flattened tables (plan.h: kFastTab entries each)
    return (plan.h.aluClass == ALU_INT64 || plan.h.aluClass == ALU_F32) && (plan.h.sampleInt || plan.h.aluClass == ALU_F32) && (plan.h.aluClass == ALU_INT64 || (plan.h.nRaw == 0 && plan.h.nMemCopy == 0)) && plan.h.nChains > 0 && plan.h.nOut > 0 && plan.h.nOut <= kFastTab &&
           plan.h.nProc <= kFastTab && plan.h.nSrc <= kFastTab;
}

bool planChain2Geometry(const ChainPlan& plan, int nStreams, int numSMs, Chain2Geom* geom, ChainLane* lanesOut) {
    const int C = plan.h.nChains;
    // sections per lane: the largest K in {4,2,1} (default 2) that divides every cascade (override: AVDSP_B200_K)
    int K = envInt2("AVDSP_B200_K", 2);
    if (K != 1 && K != 2 && K != 4) K = 2;
    for (int c = 0; c < C; c++) while (plan.chains[c].nsec % K) K >>= 1;
    int NS0 = envInt2("AVDSP_B200_NS", 0);
    if (NS0 <= 0) NS0 = (nStreams + numSMs - 1) / numSMs;
    NS0 = std::max(1, std::min(NS0, 32));
    const int forceF = envInt2("AVDSP_B200_F", 0);
    int maxDelay = 0;
    for (int c = 0; c < C; c++) maxDelay = std::max(maxDelay, plan.chains[c].delayN);
    // Every feasible streams-per-CTA count is scored: time ~ waves over the SMs x (streams per CTA + 4) (the section lanes of a CTA
    // walk their streams' frames in lock step), and the helper warps must keep up with the section warps they serve -- a CTA
    // whose 31 warps are all section lanes leaves one warp to feed and drain 20+ streams.  Pass 0 demands enough helpers,
    // pass 1 (only if nothing qualified) takes whatever fits.
    bool found = false;
    long long bestCost = 0;
    Chain2Geom bestG{};
    const bool forcedNS = envInt2("AVDSP_B200_NS", 0) > 0;
    for (int pass = 0; pass < 2 && !found; pass++)
    for (int NS = NS0; NS >= 1; NS--) {
        for (int F : {32, 16}) {
            if (forceF && F != forceF) continue;
            int gm = 0;
            const int lt = packLanes2(plan, NS, K, nullptr, &gm);
            if (lt < 0) break;
            if (gm > F) continue;                                    // sink window i must lie inside tiles i-1, i
            int help = envInt2("AVDSP_B200_HW", 0);
            if (help <= 0) help = lt > 0 ? std::max(2, std::min(32 - lt / 32, (NS + 1) / 2 + 1)) : std::min(24, std::max(4, NS));
            help = std::max(1, std::min(help, 32 - lt / 32));
            const int slots = NS * C;
            Chain2Geom g{};
            g.streamsPerCta = NS; g.secPerLane = K; g.tileFrames = F; g.gmax = gm;
            g.secThreads = lt; g.helpThreads = help * 32;
            g.helpersFirst = envInt2("AVDSP_B200_HELPFIRST", 0);
            g.debugSkip = envInt2("AVDSP_B200_DEBUG_SKIP", 0);     // timing experiments only: 1 source, 2 PRNG, 4 sink are skipped (wrong output)
            g.floatFast = 1;                                       // float class: every LOAD_GAIN gain within [2^-30, 2^30] (or exactly 0)
            for (int k = 0; k < plan.h.nSrc && k < kFastTab; k++)
                if (plan.h.sKind[k] == SRC_LOAD_GAIN) {
                    const int ex = (int)(((uint32_t)plan.h.sArg[k] >> 23) & 255u);
                    if (ex != 0 && (ex < 127 - 30 || ex > 127 + 30)) g.floatFast = 0;
                }
            if (envInt2("AVDSP_B200_FLOAT_EXACT_HELPERS", 0)) g.floatFast = 0;
            int R = 2 * F;
            while (R < 2 * F + gm + maxDelay) R <<= 1;      // tails write tile i while the sink still reads window i-1
            g.postRing = R;
            g.xPitch = 2 * F + 1; g.accPitch = 2 * F + 1; g.postPitch = R + 1; g.tpdfPitch = 4 * F + 1;
            g.accStreamBytes = plan.h.nAcc * g.accPitch * 8;
            g.xStreamBytes = plan.h.nSrc * g.xPitch * 4;
            g.postStreamBytes = C * g.postPitch * 4;
            g.tpdfStreamBytes = g.tpdfPitch * 4;
            g.rawStreamBytes = 2 * F * plan.h.nIn * 4;
            size_t bytes = (size_t)NS * g.accStreamBytes;
            g.xOff = (int)bytes;    bytes += (size_t)NS * g.xStreamBytes;
            g.postOff = (int)bytes; bytes += (size_t)NS * g.postStreamBytes;
            g.tpdfOff = (int)bytes; bytes += (size_t)NS * g.tpdfStreamBytes;
            g.ridxOff = (int)bytes; bytes += (size_t)3 * slots * 4;
            g.ckOff = (int)bytes;   bytes += (size_t)6 * K * lt * 4;        // section lanes' tile-start checkpoints
            bytes = (bytes + 15) & ~(size_t)15;
            g.mbarOff = (int)bytes; bytes += (size_t)help * 2 * 8;
            bytes = (bytes + 127) & ~(size_t)127;
            g.rawOff = plan.h.nSrc > 0 ? (int)bytes : 0;          // input tiles staged by TMA (only cascades read them)
            if (plan.h.nSrc > 0) bytes += (size_t)NS * g.rawStreamBytes;
            g.smemBytes = bytes + 16;
            for (int k = 0; k < kFastTab; k++) {
                const int oc = k < plan.h.nOut ? plan.h.chainOfOut[k] : -1;
                g.outRowOff[k] = oc >= 0 ? oc * g.postPitch * 4 : 0;
                g.outPos4[k] = plan.h.outOff[k] * 4;
                g.pPostOff[k] = k < plan.h.nProc ? plan.h.pChain[k] * g.postPitch * 4 : 0;
                g.pAccOff[k] = (k < plan.h.nProc && plan.h.pAccRow[k] >= 0) ? plan.h.pAccRow[k] * g.accPitch * 8 : 0;
                g.srcXOff[k] = k * g.xPitch * 4;
            }
            if (g.secThreads + g.helpThreads <= 1024 && g.smemBytes <= 226 * 1024) {
                const int needHelp = lt > 0 ? std::max(2, (NS + 3) / 4) : 1;
                if (pass == 0 && help < needHelp && !forcedNS) break;          // too few helper warps for this many streams
                const long long ctas = (nStreams + NS - 1) / NS;
                const long long cost = ((ctas + numSMs - 1) / numSMs) * (NS + 4);  // + a CTA's fixed cost (prologue, rings, thin warps), in streams
                if (!found || cost < bestCost) { found = true; bestCost = cost; bestG = g; }
                break;                                                          // F = 32 is preferred when it fits
            }
        }
        if (found && forcedNS) break;
    }
    if (!found) return false;
    *geom = bestG;
    if (lanesOut) packLanes2(plan, bestG.streamsPerCta, K, lanesOut, nullptr);
    return true;
}

// MEM words of inlined cascades: what the producer's STORE_MEM left there = the accumulator of its last section
__global__ void k_chain2_memfix(const __grid_constant__ ChainPlan P, int* __restrict__ state, int nStreams) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= nStreams) return;
    int* st = state + (size_t)s * P.h.stateWords;
    for (int k = 0; k < P.h.nMemCopy; k++) { st[P.h.memCopyDst[k]] = st[P.h.memCopySrc[k]]; st[P.h.memCopyDst[k] + 1] = st[P.h.memCopySrc[k] + 1]; }
}

__global__ void __launch_bounds__(256) k_redo_prepare(const int* __restrict__ state, int* __restrict__ snapshot, size_t words,
                                                      int* __restrict__ flags, int nStreams, int* __restrict__ count) {
    const size_t i0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x, step = (size_t)gridDim.x * blockDim.x;
    for (size_t i = i0; i < words; i += step) snapshot[i] = state[i];
    for (size_t i = i0; i < (size_t)nStreams; i += step) flags[i] = 0;
    if (i0 == 0) *count = 0;
}
cudaError_t launchRedoPrepare(const int* state, int* snapshot, size_t words, int* flags, int nStreams, int* count, cudaStream_t stream) {
    const int blocks = (int)std::min<size_t>((words + 255) / 256, 148 * 8);
    k_redo_prepare<<<std::max(blocks, 1), 256, 0, stream>>>(state, snapshot, words, flags, nStreams, count);
    return cudaGetLastError();
}
// flagged streams of a range -> list (any order: the streams are independent), their state blocks back to the snapshot
__global__ void __launch_bounds__(256) k_redo_compact(const int* __restrict__ flags, int nStreams, int* __restrict__ list, int* __restrict__ count,
                                                      int* __restrict__ state, const int* __restrict__ snapshot, int W) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= nStreams || !flags[warp]) return;
    int pos = 0;
    if (lane == 0) pos = atomicAdd(count, 1);
    pos = __shfl_sync(0xffffffffu, pos, 0);
    if (lane == 0) list[pos] = warp;
    for (int w = lane; w < W; w += 32) state[(size_t)warp * W + w] = snapshot[(size_t)warp * W + w];
}
cudaError_t launchRedoCompact(const int* flags, int nStreams, int* list, int* count, int* state, const int* snapshot, int stateWords, cudaStream_t stream) {
    k_redo_compact<<<(nStreams * 32 + 255) / 256, 256, 0, stream>>>(flags, nStreams, list, count, state, snapshot, stateWords);
    return cudaGetLastError();
}

cudaError_t launchChain2(const ChainPlan& plan, const Chain2Geom& geom, const Chain2Args& args, cudaStream_t stream) {
    const int blocks = (args.nStreams + geom.streamsPerCta - 1) / geom.streamsPerCta;
    const int threads = geom.secThreads + geom.helpThreads;
    cudaError_t e = cudaSuccess;
#define LAUNCH2(KK, FF) do { \
    if (plan.h.aluClass == ALU_F32) { \
        e = cudaFuncSetAttribute(k_chain2<KK, FF, ALU_F32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)geom.smemBytes); \
        if (e != cudaSuccess) return e; \
        k_chain2<KK, FF, ALU_F32><<<blocks, threads, geom.smemBytes, stream>>>(plan, args, geom); \
    } else { \
        e = cudaFuncSetAttribute(k_chain2<KK, FF, ALU_INT64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)geom.smemBytes); \
        if (e != cudaSuccess) return e; \
        k_chain2<KK, FF, ALU_INT64><<<blocks, threads, geom.smemBytes, stream>>>(plan, args, geom); \
    } } while (0)
    const int key = geom.secPerLane * 100 + geom.tileFrames;
    switch (key) {
    case 432: LAUNCH2(4, 32); break;
    case 416: LAUNCH2(4, 16); break;
    case 232: LAUNCH2(2, 32); break;
    case 216: LAUNCH2(2, 16); break;
    case 132: LAUNCH2(1, 32); break;
    default:  LAUNCH2(1, 16); break;
    }
#undef LAUNCH2
    e = cudaGetLastError();
    if (e == cudaSuccess && plan.h.nMemCopy > 0 && args.nFrames > 0) {
        k_chain2_memfix<<<(args.nStreams + 127) / 128, 128, 0, stream>>>(plan, args.state, args.nStreams);
        e = cudaGetLastError();
    }
    return e;
}

} // namespace avdsp

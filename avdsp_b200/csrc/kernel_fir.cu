// kernel_fir.cu -- DSP_FIR as a time-parallel, shared-memory-tiled kernel (BASELINE config C4).
//
// Reference semantics (runtime/dsp_runtime.c:928-969 + runtime/dsp_firSTD.h:38-52): per frame the FIR opcode
// pushes x[n] into a shifting delay line and returns  y[n] = sum_{i=0}^{N-1} x[n-i] * c[i],  summed in the order
// i = 0 -> N-1.  The delay line is O(N) moves per sample on the CPU; here it never exists during a launch:
//   * one CTA owns TT = 8 * blockDim consecutive OUTPUT samples of one (stream, path); it stages the path's taps and
//     the x window [o0-N+1, o0+TT) in shared memory (history that precedes the launch comes from the per-stream state
//     block, which keeps the reference's layout st[i] = x[n-1-i]; PCM is converted by the path's LOAD/LOAD_GAIN on the
//     way in), so HBM sees every input sample ~(1 + N/TT) times and every output once;
//   * a thread computes 8 consecutive outputs with a sliding register window of x: per 8 taps it loads 8 new x
//     (2x LDS.128) and 8 taps (2x LDS.128, broadcast) for 64 multiply-accumulates;
//   * DSP_FORMAT 2: int32 x int32 -> int64 accumulation wraps mod 2^64, so any order is bit-exact; the MAC is one
//     accumulating IMAD.WIDE (quarter rate on sm_100a: the integer-pipe roofline of this kernel);
//   * DSP_FORMAT 3: the reference's order is kept per output (taps ascending), each product truncated
//     (dspMulFloatFloat == mul.rz.ftz.f32 away from the underflow range, see avdsp_dev.cuh; the decoder only routes
//     programs here whose taps / gains keep every product above 2^-121), each sum rounded to nearest: bit-exact; the
//     eight outputs of a thread are eight independent dependency chains;
//   * k_fir_state then rewrites the delay line once per launch (st[i] = x[T-1-i], older entries shifted by T).
// The fixed-point semantics are the INTENDED ones (the reference's dsp_calc_fir_int is not a convolution,
// SURVEY.md App. C #3): same structure as the float kernel on int32 x int32 -> int64, x = ALU >> 28.
#include "avdsp_dev.cuh"
#include "kernels.h"

namespace avdsp {

constexpr int kFirR = 8;          // outputs per thread
constexpr int kFirPad = 16;       // words in front of the x window (the last register-window prefetch reads them)

template <int CLS> struct FirNum;
template <> struct FirNum<ALU_INT64> { typedef long long Acc; };
template <> struct FirNum<ALU_F32>   { typedef float Acc; };

// LOAD / LOAD_GAIN followed by the FIR's input conversion (dsp_runtime.c:565-607, :958 `ALU >> DSP_MANTBQ`);
// returns the 32-bit pattern the delay line stores (int32 s.31 or float)
template <int CLS>
__device__ __forceinline__ int firSource(const FirPath& d, int sample) {
    if constexpr (CLS == ALU_INT64) {
        const long long X = d.srcKind == SRC_LOAD_GAIN ? mul32(sample, d.srcArg) : (long long)sample;
        return (int)(X >> kMantBQ);
    } else {
        const float t = i2fScaled(sample, 31);
        return __float_as_int(d.srcKind == SRC_LOAD_GAIN ? mulFF(t, __int_as_float(d.srcArg)) : t);
    }
}
// [GAIN] -> SAT0DB[_GAIN] -> STORE (dsp_runtime.c:636-640, 464-534, 610-633)
template <int CLS>
__device__ __forceinline__ int firFinish(const FirPath& d, typename FirNum<CLS>::Acc acc, int mask) {
    if constexpr (CLS == ALU_INT64) {
        long long X = acc;
        if (d.flags & PF_GAIN) X = X * (long long)d.gainBits;
        if (d.flags & PF_SAT_GAIN) { X >>= kMant; X = X * (long long)d.satGainBits; }
        return (int)sat64_031(X) & mask;
    } else {
        float X = acc;
        if (d.flags & PF_GAIN) X = __fmul_rn(X, __int_as_float(d.gainBits));
        if (d.flags & PF_SAT_GAIN) X = mulFF(X, __int_as_float(d.satGainBits));
        return f2s31SatFast(__float_as_int(X)) & mask;
    }
}

template <int CLS>
__device__ __forceinline__ void firMac(typename FirNum<CLS>::Acc& acc, int x, int c) {
    if constexpr (CLS == ALU_INT64) acc = mac32(acc, x, c);
    else acc = __fadd_rn(acc, mulFF_fast(__int_as_float(x), __int_as_float(c)));
}

// 8 taps x 8 outputs.  Output r at tap kb+jj needs x[o_r - kb - jj] = hi[r-jj] (r >= jj) or lo[8+r-jj].
template <int CLS>
__device__ __forceinline__ void firGroup(typename FirNum<CLS>::Acc (&acc)[kFirR], const int (&hi)[kFirR], const int (&lo)[kFirR],
                                         const int (&c)[kFirR]) {
#pragma unroll
    for (int jj = 0; jj < kFirR; jj++)
#pragma unroll
        for (int r = 0; r < kFirR; r++)
            firMac<CLS>(acc[r], (r >= jj) ? hi[r - jj] : lo[kFirR + r - jj], c[jj]);
}
__device__ __forceinline__ void ld8(int (&v)[kFirR], const int* p) {
    const int4 a = *reinterpret_cast<const int4*>(p), b = *reinterpret_cast<const int4*>(p + 4);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}

// TAB: the taps come from the stream's row of the per-stream FIR table (FirArgs::taps), and a stream whose flag word is set
// (FirArgs::skip, float rows with a tap the kernel cannot multiply exactly) is left to the interpreter.  A separate instance, so
// that the shared-taps kernel stays what it was.
template <int CLS, bool TAB>
__global__ void __launch_bounds__(256)
k_fir(const __grid_constant__ FirPlan P, const FirArgs A, const int nTiles, const int H) {
    extern __shared__ __align__(16) int fir_sm[];
    typedef typename FirNum<CLS>::Acc Acc;
    const int TT = (int)blockDim.x * kFirR;
    int b = (int)blockIdx.x;
    const int tile = b % nTiles; b /= nTiles;
    const int path = b % P.nPaths;
    const int stream = b / P.nPaths;
    if (TAB && A.skip && A.skip[stream]) return;
    const FirPath& d = P.paths[path];
    int* cs = fir_sm;                              // [H] taps, zero-padded to a multiple of 16
    int* xs = fir_sm + H + kFirPad;                // [H + TT] x window: xs[jp] = x[o0 - H + jp]
    const int N = d.length;
    const int tid = (int)threadIdx.x;
    const int* taps = TAB ? A.taps + (size_t)stream * A.tapPitch + d.tapCol : A.bigPool + d.tapsOff;
    for (int k = tid; k < H; k += (int)blockDim.x) cs[k] = k < N ? taps[k] : 0;
    const int o0 = tile * TT;
    const int* in = A.in + (size_t)stream * A.inStreamStride + (size_t)(d.srcCh >= 0 ? d.srcCh : 0) * A.inChStride;
    const int* st = A.state + (size_t)stream * P.stateWords + d.stateOff;
    for (int jp = tid; jp < H + TT; jp += (int)blockDim.x) {
        const int j = o0 - H + jp;
        int v = 0;
        if (j >= 0) { if (j < A.nFrames) v = firSource<CLS>(d, d.srcCh >= 0 ? in[(size_t)j * A.inFrameStride] : 0); }
        else { const int si = -1 - j; if (si < N) v = st[si]; }
        xs[jp] = v;
    }
    if (tid < kFirPad) fir_sm[H + tid] = 0;
    __syncthreads();

    Acc acc[kFirR];
#pragma unroll
    for (int r = 0; r < kFirR; r++) acc[r] = 0;
    const int* xp = xs + H + tid * kFirR;          // the thread's own 8 samples; earlier samples lie below
    int wa[kFirR], wb[kFirR], c[kFirR];
    ld8(wa, xp); ld8(wb, xp - kFirR);
    for (int kb = 0; kb < H; kb += 2 * kFirR) {
        ld8(c, cs + kb);
        firGroup<CLS>(acc, wa, wb, c);
        ld8(wa, xp - kb - 2 * kFirR);
        ld8(c, cs + kb + kFirR);
        firGroup<CLS>(acc, wb, wa, c);
        ld8(wb, xp - kb - 3 * kFirR);
    }

    int* out = A.out + (size_t)stream * A.outStreamStride;
#pragma unroll
    for (int r = 0; r < kFirR; r++) {
        const int o = o0 + tid * kFirR + r;
        if (o < A.nFrames) {
            const int v = firFinish<CLS>(d, acc[r], P.storeMask);
            for (int s = 0; s < d.nStores; s++) out[(size_t)o * A.outFrameStride + (size_t)d.storeCh[s] * A.outChStride] = v;
            if (path == 0)
                for (int u = 0; u < P.nUnwritten; u++) out[(size_t)o * A.outFrameStride + (size_t)P.unwritten[u] * A.outChStride] = 0;
        }
    }
}

// delay line after T frames: st[i] = x[T-1-i] for i < T, the older entries move up by T (dsp_firSTD.h:43-47 applied T times)
template <int CLS, bool TAB>
__global__ void __launch_bounds__(256)
k_fir_state(const __grid_constant__ FirPlan P, const FirArgs A) {
    extern __shared__ __align__(16) int fir_sm[];
    const int path = (int)blockIdx.x % P.nPaths, stream = (int)blockIdx.x / P.nPaths;
    if (TAB && A.skip && A.skip[stream]) return;
    const FirPath& d = P.paths[path];
    const int N = d.length, T = A.nFrames;
    const int* in = A.in + (size_t)stream * A.inStreamStride + (size_t)(d.srcCh >= 0 ? d.srcCh : 0) * A.inChStride;
    int* st = A.state + (size_t)stream * P.stateWords + d.stateOff;
    for (int i = (int)threadIdx.x; i < N; i += (int)blockDim.x)
        fir_sm[i] = i < T ? firSource<CLS>(d, d.srcCh >= 0 ? in[(size_t)(T - 1 - i) * A.inFrameStride] : 0) : st[i - T];
    __syncthreads();
    for (int i = (int)threadIdx.x; i < N; i += (int)blockDim.x) st[i] = fir_sm[i];
}

template <int CLS, bool TAB>
static cudaError_t launchFirT(const FirPlan& P, const FirArgs& A, cudaStream_t stream, int* launches) {
    const int H = (P.maxLen + 15) & ~15;
    int threads = (A.nFrames + kFirR - 1) / kFirR;
    threads = threads >= 256 ? 256 : ((threads + 31) & ~31);
    const int TT = threads * kFirR;
    const int nTiles = (A.nFrames + TT - 1) / TT;
    const size_t smem = (size_t)(2 * H + kFirPad + TT) * sizeof(int);
    cudaError_t e = cudaFuncSetAttribute(k_fir<CLS, TAB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    const long long ctas = (long long)nTiles * P.nPaths * A.nStreams;
    if (ctas > 0x7FFFFFFFll) return cudaErrorInvalidConfiguration;
    k_fir<CLS, TAB><<<(unsigned)ctas, threads, smem, stream>>>(P, A, nTiles, H);
    e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    if (launches) *launches = 2;
    return launchFirState(P, A, stream);
}

cudaError_t launchFirState(const FirPlan& P, const FirArgs& A, cudaStream_t stream) {
    const unsigned grid = (unsigned)(P.nPaths * A.nStreams);
    const size_t smem = (size_t)P.maxLen * sizeof(int);
    if (A.taps) {
        if (P.aluClass == ALU_INT64) k_fir_state<ALU_INT64, true><<<grid, 256, smem, stream>>>(P, A);
        else k_fir_state<ALU_F32, true><<<grid, 256, smem, stream>>>(P, A);
    } else {
        if (P.aluClass == ALU_INT64) k_fir_state<ALU_INT64, false><<<grid, 256, smem, stream>>>(P, A);
        else k_fir_state<ALU_F32, false><<<grid, 256, smem, stream>>>(P, A);
    }
    return cudaGetLastError();
}

cudaError_t launchFir(const FirPlan& plan, const FirArgs& args, int numSMs, cudaStream_t stream, int* launches) {
    (void)numSMs;
    if (args.taps) {
        if (plan.aluClass == ALU_INT64) return launchFirT<ALU_INT64, true>(plan, args, stream, launches);
        return launchFirT<ALU_F32, true>(plan, args, stream, launches);
    }
    if (plan.aluClass == ALU_INT64) return launchFirT<ALU_INT64, false>(plan, args, stream, launches);
    return launchFirT<ALU_F32, false>(plan, args, stream, launches);
}

} // namespace avdsp

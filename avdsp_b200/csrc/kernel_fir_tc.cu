// kernel_fir_tc.cu -- DSP_FIR as a Toeplitz GEMM on the 5th-generation tensor cores (tcgen05 + TMEM), sm_100a.
//
// A long FIR shared by many streams IS a dense contraction:  Y[o, s] = sum_j C[o, j] * X[j, s]  with C[o, j] = c[o - j]
// (the taps as a banded Toeplitz matrix, identical for every stream and every output block) and X[j, s] = x_s[j]
// (time x streams).  One CTA computes a 128-output x NS-stream block: M = 128 output samples, N = NS streams,
// K = the Hc + 128 input samples that block can see, walked in stages of 128 (int8) or 64 (TF32) bytes of K.
//
//   * KIND_I8 -- DSP_FORMAT 2, BIT-EXACT.  int32 taps and samples are split into four 8-bit limbs (top limb signed,
//     the others unsigned): x = sum_i x_i 2^(8i).  The 16 limb products run as kind::i8 MMAs with int32 accumulators
//     in TMEM; products with the same i+j share an accumulator (7 accumulators x 64 streams = 448 TMEM columns), and
//     |acc| <= 4 * 255 * 255 * 8192 < 2^31, so nothing overflows.  The epilogue recombines  y = sum_s acc_s << 8s  in
//     wrapping int64 -- exactly the reference's int64 accumulation (runtime/dsp_firSTD.h, intended semantics) -- and
//     applies the path's [GAIN] -> SAT0DB[_GAIN] -> STORE.  16 int8 MACs replace one quarter-rate IMAD.WIDE.
//   * KIND_TF32 -- DSP_FORMAT 3 under a STATED TOLERANCE (not the reference's summation order): 3xTF32 split,
//     x = x_hi + x_lo, c = c_hi + c_lo, products hi*hi + hi*lo + lo*hi accumulated in fp32 in TMEM.  Opt-in
//     (AVDSP_B200_KERNEL_FIR_TC); the exact float kernel (kernel_fir.cu) stays the default.
//
// Operands reach shared memory as 1-D bulk copies (cp.async.bulk + mbarrier) of blobs that are ALREADY in the
// canonical K-major swizzled layout the MMA descriptors expect (SWIZZLE_128B for the int8 planes, 2 stages of 96 KB;
// SWIZZLE_64B for TF32, 4 stages of 48 KB -- measured: 8.35 vs 8.81 ms and 5.10 vs 5.32 ms per C4 step): the taps blobs are built once on the host when the
// program is loaded (firTcBuildTaps), the sample blobs by k_firtc_pack (PCM -> LOAD/LOAD_GAIN -> limbs / hi+lo, with
// the delay-line history in front).  Warp roles: warp 0 producer, warp 1 MMA issuer (one elected thread) + TMEM
// allocation, warps 2-5 epilogue (tcgen05.ld -> registers -> global).
#include "avdsp_dev.cuh"
#include "kernels.h"
#include <cstring>
#include <vector>

namespace avdsp {

namespace {

constexpr int kTcM = 128;                 // outputs per block
constexpr int kTcSmem = 196608;           // operand ring: kStages x (A planes + B planes of one K stage)
constexpr int kTcThreads = 192;
#ifndef AVDSP_FIRTC_ROWB_I8
#define AVDSP_FIRTC_ROWB_I8 128
#endif
#ifndef AVDSP_FIRTC_ROWB_TF32
#define AVDSP_FIRTC_ROWB_TF32 64
#endif

// rowB: bytes of K per operand row and stage = the swizzle span (128: SWIZZLE_128B, 64: SWIZZLE_64B).  Shorter rows mean
// smaller stages and a deeper bulk-copy pipeline for the same shared memory (-DAVDSP_FIRTC_ROWB_I8/_TF32=64|128 for A/B runs).
template <int KIND> struct TcCfg;
template <> struct TcCfg<FIRTC_I8> {
    static constexpr int planes = 4, NS = 64, elemBytes = 1, nAcc = 7, tmemCols = 512, rowB = AVDSP_FIRTC_ROWB_I8;
};
template <> struct TcCfg<FIRTC_TF32> {
    static constexpr int planes = 2, NS = 256, elemBytes = 4, nAcc = 1, tmemCols = 256, rowB = AVDSP_FIRTC_ROWB_TF32;
};
// PER: the per-stream form (k_firtc<FIRTC_I8, true>): a B plane slot holds its NS rows at the swizzle phase of the first chunk,
// so it is one 1 KB atom longer than the rows it holds, and the ring is two such stages
constexpr int kTcSmemPer = 204800;
template <int KIND, bool PER = false> struct TcGeo {
    typedef TcCfg<KIND> C;
    static constexpr int E = C::rowB / C::elemBytes;                       // samples of K per stage
    static constexpr int aBlob = kTcM * C::rowB, bBlob = C::NS * C::rowB;  // one plane of one stage
    static constexpr int bSlot = PER ? bBlob + 1024 : bBlob;               // shared-memory slot of one B plane
    static constexpr int stageBytes = C::planes * (aBlob + bSlot);
    static constexpr int txBytes = C::planes * (aBlob + bBlob);            // bytes the bulk copies of one stage bring in
    static constexpr int stages = (PER ? kTcSmemPer : kTcSmem) / stageBytes;
};

// byte offset of (row, byteInRow) inside a [rows][rowB] K-major tile in the canonical swizzled layout: 8-row atoms of
// 8*rowB bytes; the 16-byte chunk index is XORed with the row bits the hardware swizzle uses (Swizzle<3,4,3> / <2,4,3>)
__host__ __device__ __forceinline__ unsigned swz(unsigned rowB, unsigned row, unsigned b) {
    if (rowB == 128) return (row >> 3) * 1024u + (row & 7u) * 128u + ((((b >> 4) ^ row) & 7u) << 4) + (b & 15u);
    return (row >> 3) * 512u + (row & 7u) * 64u + ((((b >> 4) ^ (row >> 1)) & 3u) << 4) + (b & 15u);
}

__device__ __forceinline__ unsigned smemAddr(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbarInit(unsigned bar, int count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(bar), "r"(count) : "memory"); }
__device__ __forceinline__ void mbarExpectTx(unsigned bar, unsigned bytes) { asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(bar), "r"(bytes) : "memory"); }
__device__ __forceinline__ void tmaLoad1D(unsigned dst, const void* src, unsigned bytes, unsigned bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" :: "r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void mbarWait(unsigned bar, unsigned parity) {
    asm volatile("{\n.reg .pred P1;\nTCW_LOOP:\nmbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n@P1 bra TCW_DONE;\nbra TCW_LOOP;\nTCW_DONE:\n}" :: "r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ bool electOne() {
    unsigned pred;
    asm volatile("{\n.reg .pred P;\nelect.sync _|P, 0xffffffff;\nselp.u32 %0, 1, 0, P;\n}" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void tcFenceBefore() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcFenceAfter()  { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcCommit(unsigned bar) { asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(bar) : "memory"); }

// shared-memory matrix descriptor, K-major, swizzled: rows rowB bytes apart inside an 8-row atom, atoms 8*rowB bytes apart
// (SBO), version 1 (sm_100), layout type 2 = SWIZZLE_128B / 4 = SWIZZLE_64B
template <int ROWB>
__device__ __forceinline__ unsigned long long smemDesc(unsigned addr) {
    constexpr unsigned long long sbo = (8ull * ROWB) >> 4, lt = ROWB == 128 ? 2ull : 4ull;
    return (unsigned long long)((addr >> 4) & 0x3FFFu) | (1ull << 16) | (sbo << 32) | (1ull << 46) | (lt << 61);
}

template <int KIND>
__device__ __forceinline__ void mma(unsigned dTmem, unsigned long long aDesc, unsigned long long bDesc, unsigned idesc, unsigned accumulate) {
    if constexpr (KIND == FIRTC_I8)
        asm volatile("{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n}" :: "r"(dTmem), "l"(aDesc), "l"(bDesc), "r"(idesc), "r"(accumulate) : "memory");
    else
        asm volatile("{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n}" :: "r"(dTmem), "l"(aDesc), "l"(bDesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tmemLd8(unsigned taddr, int (&v)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]) : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmemLdWait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// instruction descriptor: dense, K-major A and B, M = 128, N = NS
template <int KIND>
__device__ __forceinline__ unsigned instrDesc(int aSigned, int bSigned) {
    constexpr unsigned NS = TcCfg<KIND>::NS;
    unsigned d = ((NS >> 3) << 17) | ((unsigned)(kTcM >> 4) << 24);
    if constexpr (KIND == FIRTC_I8) d |= (2u << 4) | ((unsigned)aSigned << 7) | ((unsigned)bSigned << 10);      // D = S32, A/B u8 or s8
    else d |= (1u << 4) | (2u << 7) | (2u << 10);                                                                 // D = F32, A/B TF32
    return d;
}

// ---- source / finish: the same conversions as kernel_fir.cu ------------------------------------------------
template <int KIND>
__device__ __forceinline__ int tcSource(const FirPath& d, int sample) {
    if constexpr (KIND == FIRTC_I8) {
        const long long X = d.srcKind == SRC_LOAD_GAIN ? mul32(sample, d.srcArg) : (long long)sample;
        return (int)(X >> kMantBQ);
    } else {
        const float t = i2fScaled(sample, 31);
        return __float_as_int(d.srcKind == SRC_LOAD_GAIN ? mulFF(t, __int_as_float(d.srcArg)) : t);
    }
}
__device__ __forceinline__ int tcFinishI(const FirPath& d, long long X, int mask) {
    if (d.flags & PF_GAIN) X = X * (long long)d.gainBits;
    if (d.flags & PF_SAT_GAIN) { X >>= kMant; X = X * (long long)d.satGainBits; }
    return (int)sat64_031(X) & mask;
}
__device__ __forceinline__ int tcFinishF(const FirPath& d, float X, int mask) {
    if (d.flags & PF_GAIN) X = __fmul_rn(X, __int_as_float(d.gainBits));
    if (d.flags & PF_SAT_GAIN) X = mulFF(X, __int_as_float(d.satGainBits));
    return f2s31SatFast(__float_as_int(X)) & mask;      // hardware convert for |X| in [2^-31, 1), the restatement otherwise
}

// ---- pack: PCM (+ delay-line history) -> pre-swizzled B blobs ---------------------------------------------------
// element index e in [0, Hc + Tpad) <-> time t = e - Hc; blob (path, plane, streamTile, e / E) holds NS rows x 128 B
template <int KIND>
__global__ void __launch_bounds__(256)
k_firtc_pack(const __grid_constant__ FirPlan P, const FirArgs A, unsigned char* __restrict__ ws, const int Hc, const int Tpad, const int nStreamTiles) {
    typedef TcCfg<KIND> C;
    const int quadsPerRow = (Hc + Tpad) / 4;
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long total = (long long)P.nPaths * nStreamTiles * C::NS * quadsPerRow;
    if (gid >= total) return;
    const int q = (int)(gid % quadsPerRow);
    long long r = gid / quadsPerRow;
    const int row = (int)(r % C::NS); r /= C::NS;
    const int tile = (int)(r % nStreamTiles);
    const int path = (int)(r / nStreamTiles);
    const int stream = tile * C::NS + row;
    const FirPath& d = P.paths[path];
    int x[4] = {0, 0, 0, 0};
    if (stream < A.nStreams) {
        const int* in = A.in + (size_t)stream * A.inStreamStride + (size_t)(d.srcCh >= 0 ? d.srcCh : 0) * A.inChStride;
        const int* st = A.state + (size_t)stream * P.stateWords + d.stateOff;
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const int t = 4 * q + k - Hc;
            if (t >= 0) { if (t < A.nFrames) x[k] = tcSource<KIND>(d, d.srcCh >= 0 ? in[(size_t)t * A.inFrameStride] : 0); }
            else { const int si = -1 - t; if (si < d.length) x[k] = st[si]; }
        }
    }
    typedef TcGeo<KIND> G;
    const int e = 4 * q;
    const int nTimeTiles = (Hc + Tpad) / G::E;
    const size_t blobBytes = (size_t)G::bBlob;
    const unsigned inTile = swz(C::rowB, (unsigned)row, (unsigned)((e % G::E) * C::elemBytes));
#pragma unroll
    for (int pl = 0; pl < C::planes; pl++) {
        unsigned char* blob = ws + ((((size_t)path * C::planes + pl) * nStreamTiles + tile) * nTimeTiles + e / G::E) * blobBytes;
        if constexpr (KIND == FIRTC_I8) {
            const unsigned w = ((unsigned)(x[0] >> (8 * pl)) & 255u) | (((unsigned)(x[1] >> (8 * pl)) & 255u) << 8) |
                               (((unsigned)(x[2] >> (8 * pl)) & 255u) << 16) | (((unsigned)(x[3] >> (8 * pl)) & 255u) << 24);
            *reinterpret_cast<unsigned*>(blob + inTile) = w;
        } else {
            int4 v;
            int* vp = &v.x;
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const int hi = x[k] & (int)0xFFFFE000;
                if (pl == 0) vp[k] = hi;
                else vp[k] = __float_as_int(__fsub_rn(__int_as_float(x[k]), __int_as_float(hi))) & (int)0xFFFFE000;
            }
            *reinterpret_cast<int4*>(blob + inTile) = v;
        }
    }
}

// ---- the GEMM ---------------------------------------------------------------------------------------------------
// PER (FIRTC_I8 only): taps of the stream's own (device-built) Toeplitz planes; the N index runs over NS consecutive 128-frame
// output blocks of one stream instead of over streams.  blockIdx = (group of NS blocks, tile = the call's stream, path).
template <int KIND, bool PER>
__global__ void __launch_bounds__(kTcThreads, 1)
k_firtc(const __grid_constant__ FirPlan P, const FirArgs A, const unsigned char* __restrict__ taps, const unsigned char* __restrict__ ws,
        const int Hc, const int Tpad, const int nStreamTiles) {
    typedef TcCfg<KIND> C;
    typedef TcGeo<KIND, PER> G;
    constexpr int kTcStages = G::stages, kStageBytes = G::stageBytes;
    extern __shared__ __align__(1024) unsigned char tc_sm[];
    __shared__ __align__(8) unsigned long long bars[2 * kTcStages + 1];
    __shared__ unsigned tmemBase;
    const int warp = (int)threadIdx.x >> 5, lane = (int)threadIdx.x & 31;
    const int Q = (int)blockIdx.x, tile = (int)blockIdx.y, path = (int)blockIdx.z;
    const int nStages = (Hc + kTcM) / G::E;
    const int nTimeTiles = (Hc + Tpad) / G::E;
    const unsigned smBase = (smemAddr(tc_sm) + 1023u) & ~1023u;
    const unsigned barFull = smemAddr(&bars[0]), barEmpty = smemAddr(&bars[kTcStages]), barAcc = smemAddr(&bars[2 * kTcStages]);
    constexpr unsigned aBlob = G::aBlob, bBlob = G::bBlob, bSlot = G::bSlot;

    if (warp == 0 && lane == 0) {
        for (int s = 0; s < kTcStages; s++) { mbarInit(barFull + 8 * s, 1); mbarInit(barEmpty + 8 * s, 1); }
        mbarInit(barAcc, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smemAddr(&tmemBase)), "r"((unsigned)C::tmemCols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tcFenceBefore();
    __syncthreads();
    tcFenceAfter();
    const unsigned tmem = tmemBase;

    if (warp == 0) {
        if (lane == 0) {
            // ===== producer: one bulk copy per operand plane and stage =====
            const unsigned char* aSrc = taps + ((PER ? (size_t)tile * P.nPaths : 0) + path) * C::planes * nStages * aBlob;
            const unsigned char* bSrc = PER ? ws + (((size_t)path * C::planes) * nStreamTiles + tile) * (size_t)(Hc + Tpad)
                                            : ws + (((size_t)path * C::planes) * nStreamTiles + tile) * nTimeTiles * (size_t)bBlob;
            const size_t bPlaneStride = PER ? (size_t)nStreamTiles * (Hc + Tpad) : (size_t)nStreamTiles * nTimeTiles * bBlob;
            const int tau0 = Q * (PER ? C::NS : kTcM / G::E);
            for (int st = 0; st < nStages; st++) {
                const int slot = st % kTcStages;
                mbarWait(barEmpty + 8 * slot, (((unsigned)st / kTcStages) & 1u) ^ 1u);
                mbarExpectTx(barFull + 8 * slot, (unsigned)G::txBytes);
                const unsigned dst = smBase + (unsigned)slot * kStageBytes;
#pragma unroll
                for (int pl = 0; pl < C::planes; pl++) {
                    tmaLoad1D(dst + pl * aBlob, aSrc + ((size_t)pl * nStages + st) * aBlob, aBlob, barFull + 8 * slot);
                    if constexpr (PER)      // NS consecutive chunks (rows) of the stream's chunk plane, from chunk tau0 + st, at its phase
                        tmaLoad1D(dst + C::planes * aBlob + pl * bSlot + (unsigned)((tau0 + st) & 7) * C::rowB,
                                  bSrc + pl * bPlaneStride + (size_t)(tau0 + st) * C::rowB, bBlob, barFull + 8 * slot);
                    else
                        tmaLoad1D(dst + C::planes * aBlob + pl * bBlob, bSrc + pl * bPlaneStride + (size_t)(tau0 + st) * bBlob, bBlob, barFull + 8 * slot);
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer: the WHOLE warp walks the stages (uniform control flow) and one elected lane issues, so that
        // ptxas emits bare UTC*MMA instructions instead of an elect/branch wrapper around each of them =====
        for (int st = 0; st < nStages; st++) {
            const int slot = st % kTcStages;
            mbarWait(barFull + 8 * slot, ((unsigned)st / kTcStages) & 1u);
            tcFenceAfter();
            if (electOne()) {
                const unsigned aBase = smBase + (unsigned)slot * kStageBytes;
                const unsigned bBase = aBase + C::planes * aBlob + (PER ? (unsigned)(((Q * C::NS) + st) & 7) * C::rowB : 0u);
#pragma unroll
                for (int ks = 0; ks < C::rowB / 32; ks++) {                   // rowB bytes of K per stage = rowB/32 MMAs of 32 B
                    if constexpr (KIND == FIRTC_I8) {
#pragma unroll
                        for (int i = 0; i < 4; i++)
#pragma unroll
                            for (int j = 0; j < 4; j++) {
                                const int s = i + j;
                                const bool first = st == 0 && ks == 0 && i == (s > 3 ? s - 3 : 0);
                                // PER: the tile starts (st & 7) rows into a swizzle atom, its rows stored at their own phase; the
                                // swizzle follows the address bits, so the descriptor needs no base offset (measured: setting
                                // bits 49-51 to that phase gives wrong sums, leaving them 0 gives bit-exact ones)
                                const unsigned long long bDesc = PER ? smemDesc<C::rowB>(bBase + j * bSlot + ks * 32) : smemDesc<C::rowB>(bBase + j * bBlob + ks * 32);
                                mma<KIND>(tmem + (unsigned)(s * C::NS), smemDesc<C::rowB>(aBase + i * aBlob + ks * 32), bDesc,
                                          instrDesc<KIND>(i == 3, j == 3), first ? 0u : 1u);
                            }
                    } else {
                        const unsigned id = instrDesc<KIND>(0, 0);
                        // small terms first: lo*hi, hi*lo, then hi*hi
                        mma<KIND>(tmem, smemDesc<C::rowB>(aBase + aBlob + ks * 32), smemDesc<C::rowB>(bBase + ks * 32), id, (st == 0 && ks == 0) ? 0u : 1u);
                        mma<KIND>(tmem, smemDesc<C::rowB>(aBase + ks * 32), smemDesc<C::rowB>(bBase + bBlob + ks * 32), id, 1u);
                        mma<KIND>(tmem, smemDesc<C::rowB>(aBase + ks * 32), smemDesc<C::rowB>(bBase + ks * 32), id, 1u);
                    }
                }
                tcCommit(barEmpty + 8 * slot);             // frees the smem slot when these MMAs have read it
                if (st == nStages - 1) tcCommit(barAcc);   // accumulators complete
            }
            __syncwarp();
        }
    } else {
        // ===== epilogue: warps 2..5 own TMEM lane quadrants (warp % 4) =====
        const int quad = warp & 3;
        const int m = quad * 32 + lane;
        const int o = Q * kTcM + m;                     // (shared taps; PER maps frames per column below)
        const FirPath& d = P.paths[path];
        mbarWait(barAcc, 0);
        tcFenceAfter();
        const unsigned trow = tmem + ((unsigned)(quad * 32) << 16);
        const int s0 = tile * C::NS;
        for (int n0 = 0; n0 < C::NS; n0 += 8) {
            if (PER ? (Q * C::NS + n0) * kTcM >= A.nFrames : s0 + n0 >= A.nStreams) break;      // warp-uniform
            int res[8];
            if constexpr (KIND == FIRTC_I8) {
                unsigned long long y[8];
#pragma unroll
                for (int k = 0; k < 8; k++) y[k] = 0;
#pragma unroll
                for (int s = 0; s < C::nAcc; s++) {
                    int v[8];
                    tmemLd8(trow + (unsigned)(s * C::NS + n0), v);
                    tmemLdWait();
#pragma unroll
                    for (int k = 0; k < 8; k++) y[k] += (unsigned long long)(long long)v[k] << (8 * s);
                }
#pragma unroll
                for (int k = 0; k < 8; k++) res[k] = tcFinishI(d, (long long)y[k], P.storeMask);
            } else {
                int v[8];
                tmemLd8(trow + (unsigned)n0, v);
                tmemLdWait();
#pragma unroll
                for (int k = 0; k < 8; k++) res[k] = tcFinishF(d, __int_as_float(v[k]), P.storeMask);
            }
            if constexpr (PER) {                            // N = output blocks of stream `tile`: frame 128 * block + m
#pragma unroll
                for (int k = 0; k < 8; k++) {
                    const int f = (Q * C::NS + n0 + k) * kTcM + m;
                    if (f < A.nFrames) {
                        int* out = A.out + (size_t)tile * A.outStreamStride + (size_t)f * A.outFrameStride;
                        for (int q = 0; q < d.nStores; q++) out[(size_t)d.storeCh[q] * A.outChStride] = res[k];
                        if (path == 0) for (int u = 0; u < P.nUnwritten; u++) out[(size_t)P.unwritten[u] * A.outChStride] = 0;
                    }
                }
            } else if (o < A.nFrames) {
#pragma unroll
                for (int k = 0; k < 8; k++) {
                    const int stream = s0 + n0 + k;
                    if (stream < A.nStreams) {
                        int* out = A.out + (size_t)stream * A.outStreamStride + (size_t)o * A.outFrameStride;
                        for (int q = 0; q < d.nStores; q++) out[(size_t)d.storeCh[q] * A.outChStride] = res[k];
                        if (path == 0) for (int u = 0; u < P.nUnwritten; u++) out[(size_t)P.unwritten[u] * A.outChStride] = 0;
                    }
                }
            }
        }
    }
    tcFenceBefore();
    __syncthreads();
    if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem), "r"((unsigned)C::tmemCols) : "memory");
}

// ---- per-stream form: operands ------------------------------------------------------------------------------------
// B: one chunk plane per (path, limb plane, stream): rows = 128-sample chunks of the stream's input (element e = t + Hc, delay-line
// history in front), chunk r at r * 128 bytes, swizzled at its own phase r & 7 -- so that any NS consecutive rows copied to the
// matching phase of a shared-memory atom form a valid SWIZZLE_128B tile (swz(128, r, b) = r * 128 + the swizzled byte)
__global__ void __launch_bounds__(256)
k_firtc_pack_per(const __grid_constant__ FirPlan P, const FirArgs A, unsigned char* __restrict__ ws, const int Hc, const int Tpad) {
    const int quadsPerRow = (Hc + Tpad) / 4;
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= (long long)P.nPaths * A.nStreams * quadsPerRow) return;
    const int q = (int)(gid % quadsPerRow);
    const long long r = gid / quadsPerRow;
    const int stream = (int)(r % A.nStreams), path = (int)(r / A.nStreams);
    const FirPath& d = P.paths[path];
    const int* in = A.in + (size_t)stream * A.inStreamStride + (size_t)(d.srcCh >= 0 ? d.srcCh : 0) * A.inChStride;
    const int* st = A.state + (size_t)stream * P.stateWords + d.stateOff;
    int x[4];
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const int t = 4 * q + k - Hc;
        x[k] = 0;
        if (t >= 0) { if (t < A.nFrames) x[k] = tcSource<FIRTC_I8>(d, d.srcCh >= 0 ? in[(size_t)t * A.inFrameStride] : 0); }
        else { const int si = -1 - t; if (si < d.length) x[k] = st[si]; }
    }
    const int e = 4 * q;
    const size_t planeBytes = (size_t)(Hc + Tpad);
    const unsigned off = swz(128u, (unsigned)(e >> 7), (unsigned)(e & 127));
#pragma unroll
    for (int pl = 0; pl < 4; pl++) {
        unsigned char* plane = ws + (((size_t)path * 4 + pl) * A.nStreams + stream) * planeBytes;
        const unsigned w = ((unsigned)(x[0] >> (8 * pl)) & 255u) | (((unsigned)(x[1] >> (8 * pl)) & 255u) << 8) |
                           (((unsigned)(x[2] >> (8 * pl)) & 255u) << 16) | (((unsigned)(x[3] >> (8 * pl)) & 255u) << 24);
        *reinterpret_cast<unsigned*>(plane + off) = w;
    }
}

// A: every stream's own Toeplitz limb planes from its row of the FIR table, the device counterpart of firTcBuildTaps:
// blob (stream, path, plane, stage) = [128 rows m][128 B], A[m, k] = c[m + Hc - k].  One thread: 4 consecutive k of one row.
__global__ void __launch_bounds__(256)
k_firtc_build_taps(const __grid_constant__ FirPlan P, const int* __restrict__ tab, const int nCols, const int nStreams, const int Hc,
                   unsigned char* __restrict__ out) {
    const int nStages = (Hc + kTcM) / 128;
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= (long long)nStreams * P.nPaths * nStages * kTcM * 32) return;
    const int w = (int)(gid & 31), m = (int)((gid >> 5) % kTcM);
    long long r = gid / (32 * kTcM);
    const int stg = (int)(r % nStages); r /= nStages;
    const int path = (int)(r % P.nPaths), stream = (int)(r / P.nPaths);
    const FirPath& d = P.paths[path];
    const int* row = tab + (size_t)stream * nCols + d.tapCol;
    int c[4];
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const int idx = m + Hc - (stg * 128 + 4 * w + k);
        c[k] = (idx >= 0 && idx < d.length) ? row[idx] : 0;
    }
    const unsigned off = swz(128u, (unsigned)m, (unsigned)(4 * w));
#pragma unroll
    for (int pl = 0; pl < 4; pl++) {
        const unsigned v = ((unsigned)(c[0] >> (8 * pl)) & 255u) | (((unsigned)(c[1] >> (8 * pl)) & 255u) << 8) |
                           (((unsigned)(c[2] >> (8 * pl)) & 255u) << 16) | (((unsigned)(c[3] >> (8 * pl)) & 255u) << 24);
        *reinterpret_cast<unsigned*>(out + ((((size_t)stream * P.nPaths + path) * 4 + pl) * nStages + stg) * (size_t)(kTcM * 128) + off) = v;
    }
}

} // namespace

// ---- host side ------------------------------------------------------------------------------------------------------
int firTcHistory(const FirPlan& P) { return (P.maxLen + 127) & ~127; }

static int firTcRowB(int kind) { return kind == FIRTC_I8 ? TcCfg<FIRTC_I8>::rowB : TcCfg<FIRTC_TF32>::rowB; }

// Taps as pre-swizzled A blobs: A[m, k] = c[m + Hc - k] for stage st = k / E, one [128 rows x rowB] blob per (path, plane, stage)
void firTcBuildTaps(const FirPlan& P, int kind, const int32_t* bigPool, std::vector<unsigned char>* out) {
    const int Hc = firTcHistory(P);
    const int rowB = firTcRowB(kind);
    const int planes = kind == FIRTC_I8 ? 4 : 2, eb = kind == FIRTC_I8 ? 1 : 4, E = rowB / eb;
    const int nStages = (Hc + kTcM) / E;
    const size_t blobBytes = (size_t)kTcM * rowB;
    out->assign((size_t)P.nPaths * planes * nStages * blobBytes, 0);
    for (int p = 0; p < P.nPaths; p++) {
        const FirPath& d = P.paths[p];
        for (int pl = 0; pl < planes; pl++)
            for (int st = 0; st < nStages; st++) {
                unsigned char* blob = out->data() + (((size_t)p * planes + pl) * nStages + st) * blobBytes;
                for (int m = 0; m < kTcM; m++)
                    for (int kk = 0; kk < E; kk++) {
                        const int idx = m + Hc - (st * E + kk);
                        if (idx < 0 || idx >= d.length) continue;
                        const int32_t c = bigPool[d.tapsOff + idx];
                        unsigned char* dst = blob + swz((unsigned)rowB, (unsigned)m, (unsigned)(kk * eb));
                        if (kind == FIRTC_I8) *dst = (unsigned char)((uint32_t)(c >> (8 * pl)) & 255u);
                        else {
                            const int32_t hi = c & (int32_t)0xFFFFE000;
                            int32_t v = hi;
                            if (pl == 1) { float fc, fh; memcpy(&fc, &c, 4); memcpy(&fh, &hi, 4); const float lo = fc - fh; memcpy(&v, &lo, 4); v &= (int32_t)0xFFFFE000; }
                            memcpy(dst, &v, 4);
                        }
                    }
            }
    }
}

size_t firTcWorkspaceBytes(const FirPlan& P, int kind, int nStreams, int nFrames) {
    const int Hc = firTcHistory(P), Tpad = (nFrames + kTcM - 1) / kTcM * kTcM;
    const int NS = kind == FIRTC_I8 ? 64 : 256, planes = kind == FIRTC_I8 ? 4 : 2, eb = kind == FIRTC_I8 ? 1 : 4;
    const int tiles = (nStreams + NS - 1) / NS;
    return (size_t)P.nPaths * planes * tiles * NS * (size_t)(Hc + Tpad) * eb;
}

template <int KIND>
static cudaError_t launchFirTcT_(const FirPlan& P, const FirArgs& A, const unsigned char* dTaps, unsigned char* ws, cudaStream_t stream) {
    typedef TcCfg<KIND> C;
    const int Hc = firTcHistory(P), Tpad = (A.nFrames + kTcM - 1) / kTcM * kTcM;
    const int tiles = (A.nStreams + C::NS - 1) / C::NS;
    const long long quads = (long long)P.nPaths * tiles * C::NS * ((Hc + Tpad) / 4);
    k_firtc_pack<KIND><<<(unsigned)((quads + 255) / 256), 256, 0, stream>>>(P, A, ws, Hc, Tpad, tiles);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    const size_t smem = (size_t)TcGeo<KIND>::stages * TcGeo<KIND>::stageBytes + 1024;
    e = cudaFuncSetAttribute(k_firtc<KIND, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    if (tiles > 65535 || P.nPaths > 65535) return cudaErrorInvalidConfiguration;
    k_firtc<KIND, false><<<dim3((unsigned)(Tpad / kTcM), (unsigned)tiles, (unsigned)P.nPaths), kTcThreads, smem, stream>>>(P, A, dTaps, ws, Hc, Tpad, tiles);
    return cudaGetLastError();
}

cudaError_t launchFirTc(const FirPlan& plan, int kind, const FirArgs& args, const unsigned char* dTaps, unsigned char* workspace,
                        cudaStream_t stream, int* launches) {
    cudaError_t e = kind == FIRTC_I8 ? launchFirTcT_<FIRTC_I8>(plan, args, dTaps, workspace, stream)
                                     : launchFirTcT_<FIRTC_TF32>(plan, args, dTaps, workspace, stream);
    if (e != cudaSuccess) return e;
    e = launchFirState(plan, args, stream);
    if (launches) *launches = 3;
    return e;
}

// ---- per-stream form (DSP_FORMAT 2 with a per-stream FIR table) ------------------------------------------------------
// frames are padded to whole groups of NS = 64 output blocks (8192 frames): one CTA = 128 outputs x 64 blocks of one stream
static int firTcPerTpad(int nFrames) { const int g = TcCfg<FIRTC_I8>::NS * kTcM; return (nFrames + g - 1) / g * g; }

size_t firTcPerTapsBytes(const FirPlan& P, int nStreams) {
    return (size_t)nStreams * P.nPaths * 4 * ((firTcHistory(P) + kTcM) / 128) * (size_t)(kTcM * 128);
}
size_t firTcPerWorkspaceBytes(const FirPlan& P, int nStreams, int nFrames) {
    return (size_t)P.nPaths * 4 * nStreams * (size_t)(firTcHistory(P) + firTcPerTpad(nFrames));
}
cudaError_t launchFirTcBuildTaps(const FirPlan& P, const int* tab, int nCols, int nStreams, unsigned char* out, cudaStream_t stream) {
    const long long n = (long long)nStreams * P.nPaths * ((firTcHistory(P) + kTcM) / 128) * kTcM * 32;
    k_firtc_build_taps<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(P, tab, nCols, nStreams, firTcHistory(P), out);
    return cudaGetLastError();
}
cudaError_t launchFirTcPer(const FirPlan& P, const FirArgs& A, const unsigned char* dTaps, unsigned char* ws, cudaStream_t stream, int* launches) {
    const int Hc = firTcHistory(P), Tpad = firTcPerTpad(A.nFrames);
    const long long quads = (long long)P.nPaths * A.nStreams * ((Hc + Tpad) / 4);
    k_firtc_pack_per<<<(unsigned)((quads + 255) / 256), 256, 0, stream>>>(P, A, ws, Hc, Tpad);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    typedef TcGeo<FIRTC_I8, true> G;
    const size_t smem = (size_t)G::stages * G::stageBytes + 1024;
    e = cudaFuncSetAttribute(k_firtc<FIRTC_I8, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    if (A.nStreams > 65535 || P.nPaths > 65535) return cudaErrorInvalidConfiguration;
    // blockIdx.x fastest: the CTAs of one stream run together and read its A planes from L2
    k_firtc<FIRTC_I8, true><<<dim3((unsigned)(Tpad / (kTcM * TcCfg<FIRTC_I8>::NS)), (unsigned)A.nStreams, (unsigned)P.nPaths), kTcThreads, smem, stream>>>(
        P, A, dTaps, ws, Hc, Tpad, A.nStreams);
    e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    e = launchFirState(P, A, stream);
    if (launches) *launches = 3;
    return e;
}

} // namespace avdsp

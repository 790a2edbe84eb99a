// kernel_dag.cu -- executor for programs that route signals through the X/Y register pair: subtractive crossovers
// (`COPYXY .. DELAY .. SWAPXY .. BIQUADS .. SUBYX`: dspprogs/crossoverLV6.c, oktodac_fabriceo.c), forks (`COPYXY .. SWAPXY`:
// crossover2x2lfe.c), sums of MEM words (`LOAD_MEM; LOAD_MEM; ADDXY`), cascades handed on through MEM words.  Fixed point
// (DSP_FORMAT 2), bit-exact (dsp_runtime.c:337-405, 565-640, 726-849; dsp_biquadSTD.h:25-77).
//
// Such a program is not a set of independent chains (kernel_chain2/3.cu): a path may start from a combination of what other
// paths computed in the SAME frame.  The decoder (decoder.cpp::buildDagPlan) executes X/Y symbolically and emits a small DAG
// whose nodes are   expression over operands -> [biquad cascade] -> [gain / saturate / dither -> delay -> stores]   (plan.h).
//
// Mapping.  One CTA owns NS streams for the whole launch; lane = stream, warp = node: a node's cascade state (accumulator,
// x1 x2 y1 y2 per section) and coefficients stay in registers for the launch, and a warp's work is uniform.  Nodes that
// depend on each other are pipelined by TILES of 32 frames: a node of depth d (1 + its deepest operand node) works on tile
// i - 1 - d at iteration i, so every node of the DAG runs in every iteration and reads what its operands wrote one or more
// iterations ago; one barrier per iteration is the only synchronisation.  Values travel through per-stream rows in shared
// memory, indexed by FRAME (mod a power of two): staged input PCM, dither values, 64-bit node values (two planes), finished
// s.31 outputs.  A finished-output row doubles as the delay line of a DSP_DELAY behind the saturation (the store warps read
// it at frame - n); DSP_DELAY on a raw sample and DSP_DELAY_DP on a node value get a private row of the consuming lane.
// All delay rows are primed from the reference's rings in the state block and written back in its layout (ring index,
// stale-index case after a shortened delay included), so any split into calls and any kernel switch is invisible.
// Unlike k_chain3 the sections of a cascade are NOT skewed in time (four of a section's five MACs do not depend on the
// current input, so the chain through a cascade is one MAC + one shift per section): no lag bookkeeping between nodes.
#include "avdsp_dev.cuh"
#include "kernels.h"
#include <algorithm>
#include <cstdlib>
#include <type_traits>

namespace avdsp {
namespace {


// one reference delay ring (dsp_runtime.c:769-824: [index | line of n elements]) mapped onto a frame-indexed row:
// frame f's value sits at f & mask, the n elements the reference ring holds at launch start are "virtual frames" -n..-1
struct DagDelay {
    int n = 0, off = 0, idx0 = 0, staleIdx = -1;
    int ovLo = 0, ovHi = 0;                 // old line[n-1]: what frame n reads back in the stale-index case
};

// WORDS = 1: int32 elements (DSP_DELAY), 2: int64 (DSP_DELAY_DP: index at an odd word so that the line is 8-aligned)
template <int WORDS>
__device__ __forceinline__ void delayPrime(DagDelay& D, int n, int off, const int* __restrict__ st, int* rowLo, int* rowHi, int mask) {
    D.n = n; D.off = off; D.staleIdx = -1; D.idx0 = 0;
    if (n <= 0) return;
    const int* line = st + off + 1;
    int idx = st[off];
    // an index >= n (the host shortened the delay) is used once by the reference -- frame 0 swaps with line[idx] -- and then
    // wraps to 0: frame k >= 1 swaps with line[k-1], so frame n reads the OLD line[n-1], not frame 0's value
    const bool stale = idx >= n || idx < 0;
    if (idx < 0) idx = 0;
    for (int k = 0; k < n; k++) {
        const int e = stale ? (k == 0 ? idx : k - 1) : (idx + k >= n ? idx + k - n : idx + k);
        rowLo[(k - n) & mask] = line[e * WORDS];
        if (WORDS == 2) rowHi[(k - n) & mask] = line[e * WORDS + 1];
    }
    if (stale) { D.staleIdx = idx; D.idx0 = n - 1; D.ovLo = line[(n - 1) * WORDS]; if (WORDS == 2) D.ovHi = line[(n - 1) * WORDS + 1]; }
    else D.idx0 = idx;
}
// frame f: park the new value, hand back the one from n frames ago
template <int WORDS>
__device__ __forceinline__ long long delayStep(const DagDelay& D, int f, long long v, int* __restrict__ st, int* rowLo, int* rowHi, int mask) {
    if (D.staleIdx >= 0 && f == 0) { st[D.off + 1 + D.staleIdx * WORDS] = lo32(v); if (WORDS == 2) st[D.off + 1 + D.staleIdx * WORDS + 1] = hi32(v); }
    rowLo[f & mask] = lo32(v);
    if (WORDS == 2) rowHi[f & mask] = hi32(v);
    int lo, hi;
    if (D.staleIdx >= 0 && f == D.n) { lo = D.ovLo; hi = D.ovHi; }
    else { lo = rowLo[(f - D.n) & mask]; hi = WORDS == 2 ? rowHi[(f - D.n) & mask] : 0; }
    if (WORDS == 2) return (long long)(((unsigned long long)(unsigned)hi << 32) | (unsigned)lo);
    return (long long)lo;                  // the 32-bit ring hands (int)X back sign-extended
}
// after T frames: the ring holds frames T-n .. T-1 (virtual ones included) at (idx0 + j) mod n, the index has advanced by T
template <int WORDS>
__device__ __forceinline__ void delayWriteBack(const DagDelay& D, int T, int* __restrict__ st, const int* rowLo, const int* rowHi, int mask) {
    if (D.n <= 0 || T <= 0) return;
    int* line = st + D.off + 1;
    for (int k = 0; k < D.n; k++) {
        const long long j = (long long)T - D.n + k;
        int pos = (int)(((long long)D.idx0 + j) % D.n); if (pos < 0) pos += D.n;
        const bool ov = D.staleIdx >= 0 && j == 0;
        line[pos * WORDS] = ov ? D.ovLo : rowLo[(int)j & mask];
        if (WORDS == 2) line[pos * WORDS + 1] = ov ? D.ovHi : rowHi[(int)j & mask];
    }
    st[D.off] = (int)(((long long)D.idx0 + T) % D.n);
}

struct DagLaneCtx {
    int* blk;                               // this lane's stream block in shared memory
    int* st;                                // ... and in HBM
};

// value of one operand at frame f (warp-uniform control flow: the descriptor sits in the constant bank)
__device__ __forceinline__ long long dagOperand(const DagPlan& P, const DagGeom& G, const DagOperand& o, const DagDelay& D, int dlyOff, int dlyMask,
                                                const DagLaneCtx& C, int f, long long& muxLast) {
    switch (o.kind) {
    case OPD_RAW: {
        int smp = o.arg >= 0 ? C.blk[G.rawOff + o.arg * (G.rawMask + 1) + (f & G.rawMask)] : 0;
        if (o.delayKind == 1) smp = (int)delayStep<1>(D, f, (long long)smp, C.st, C.blk + dlyOff, nullptr, dlyMask);
        return o.hasGain ? mul32(smp, o.gain) : (long long)smp;
    }
    case OPD_NODE: {
        const int lo = C.blk[G.accLoOff[o.arg] + (f & G.accMask[o.arg])], hi = C.blk[G.accHiOff[o.arg] + (f & G.accMask[o.arg])];
        long long v = (long long)(((unsigned long long)(unsigned)hi << 32) | (unsigned)lo);
        if (o.delayKind == 2) v = delayStep<2>(D, f, v, C.st, C.blk + dlyOff, C.blk + dlyOff + dlyMask + 1, dlyMask);
        return v;
    }
    case OPD_MUX: {
        long long X = 0;
        for (int k = 0; k < o.n; k++) {
            const int ch = P.pool[o.arg + 2 * k], gain = P.pool[o.arg + 2 * k + 1];
            X = mac32(X, ch >= 0 ? C.blk[G.rawOff + ch * (G.rawMask + 1) + (f & G.rawMask)] : 0, gain);
        }
        muxLast = X;
        return X;
    }
    default: return 0;
    }
}

template <int NSEC>
__device__ __forceinline__ void dagNodeWarp(const DagPlan& P, const Chain2Args& A, const DagGeom& G, int* smem, int w, int lane) {
    const DagNode& n = P.nodes[w];
    const int NS = G.streamsPerCta, T = A.nFrames, W = P.stateWords;
    const int s0 = blockIdx.x * NS, nsHere = min(NS, A.nStreams - s0);
    const bool live = lane < nsHere;
    const int FD = G.tileFrames;
    const int nTiles = (T + FD - 1) / FD, nIter = nTiles + P.maxDepth + 2;
    DagLaneCtx C;
    C.blk = smem + (live ? lane : 0) * G.perStreamWords;
    C.st = A.state + (size_t)(s0 + (live ? lane : 0)) * W;
    // cascade state in registers.  The two history words of a section swap roles every frame (even frames: x1 = xa, x2 = xb and
    // the new x lands in xb; odd frames the other way round), so the frame loop, unrolled by two, carries no register moves
    // (ptxas emits them as IMAD.MOVs, on the very pipe the MACs run on)
    constexpr int NS_ = NSEC > 0 ? NSEC : 1;
    long long sAcc[NS_];
    int xa[NS_], xb[NS_], ya[NS_], yb[NS_];
    int cf[NS_][5];
    DagDelay da, db, dp;
    const int postMask = G.postMask[w], postOff = G.postOff[w];
    if (live) {
#pragma unroll
        for (int k = 0; k < NSEC; k++) {
            const int* q = C.st + P.pool[n.secStateOff + k];          // [acc_lo, acc_hi, x1, x2, y1, y2] (dsp_biquadSTD.h:45)
            sAcc[k] = (long long)(((unsigned long long)(unsigned)q[1] << 32) | (unsigned)q[0]);
            xa[k] = q[2]; xb[k] = q[3]; ya[k] = q[4]; yb[k] = q[5];
            sectionCoefs(P.pool + n.coefOff + 5 * k, A.coefs, A.coefPitch, P.pool[n.coefColOff + k], s0 + lane, cf[k]);
        }
        if (n.a.delayKind == 1) delayPrime<1>(da, n.a.delayN, n.a.delayOff, C.st, C.blk + G.aDlyOff[w], nullptr, G.aDlyMask[w]);
        if (n.a.delayKind == 2) delayPrime<2>(da, n.a.delayN, n.a.delayOff, C.st, C.blk + G.aDlyOff[w], C.blk + G.aDlyOff[w] + G.aDlyMask[w] + 1, G.aDlyMask[w]);
        if (n.b.delayKind == 1) delayPrime<1>(db, n.b.delayN, n.b.delayOff, C.st, C.blk + G.bDlyOff[w], nullptr, G.bDlyMask[w]);
        if (n.b.delayKind == 2) delayPrime<2>(db, n.b.delayN, n.b.delayOff, C.st, C.blk + G.bDlyOff[w], C.blk + G.bDlyOff[w] + G.bDlyMask[w] + 1, G.bDlyMask[w]);
        if (n.finKind != FIN_NONE && n.delayN > 0) {
            delayPrime<1>(dp, n.delayN, n.delayOff, C.st, C.blk + postOff, nullptr, postMask);
            // the store warps read this row: what they need to know about a stale index
            smem[G.staleOff + (w * 32 + lane) * 2] = dp.staleIdx >= 0 ? 1 : 0;
            smem[G.staleOff + (w * 32 + lane) * 2 + 1] = dp.ovLo;
        } else if (n.finKind != FIN_NONE) smem[G.staleOff + (w * 32 + lane) * 2] = 0;
    }
    // the node's description in registers (the plan sits in the constant bank, but the frame loop should not re-read it)
    const DagOperand oa = n.a, ob = n.b;
    const int comb = n.comb, postShift = n.postShift, hasPostGain = n.hasPostGain, postGain = n.postGain;
    const int exportAcc = n.exportAcc, finKind = n.finKind, finHasGain = n.finHasGain, finGain = n.finGain, satKind = n.satKind, satGain = n.satGain;
    const int aDlyOff = G.aDlyOff[w], aDlyMask = G.aDlyMask[w], bDlyOff = G.bDlyOff[w], bDlyMask = G.bDlyMask[w];
    const int accLo = G.accLoOff[w], accHi = G.accHiOff[w], accMask = G.accMask[w];
    const int tpdfOff = G.tpdfOff, tpdfMask = G.tpdfMask, tpdfShift = P.tpdfShift;
    // the common source: one input sample, LOAD or LOAD_GAIN, nothing else in front of the cascade
    const bool simpleIn = oa.kind == OPD_RAW && oa.arg >= 0 && !oa.delayKind && !comb && !postShift && !hasPostGain;
    const int* rawRow = C.blk + G.rawOff + (oa.kind == OPD_RAW && oa.arg >= 0 ? oa.arg : 0) * (G.rawMask + 1);
    const int rawMask = G.rawMask;
    long long muxLast = 0, lastAcc = 0;

    // one frame; PAR selects which of the two history register sets plays "1" this frame
    auto frame = [&](int f, auto parTag) {
        constexpr bool PAR = decltype(parTag)::value;
        long long V;
        if (simpleIn) {
            const int smp = rawRow[f & rawMask];
            V = oa.hasGain ? mul32(smp, oa.gain) : (long long)smp;
        } else {
            V = dagOperand(P, G, oa, da, aDlyOff, aDlyMask, C, f, muxLast);
            if (comb) {
                const long long B = dagOperand(P, G, ob, db, bDlyOff, bDlyMask, C, f, muxLast);
                V = comb > 0 ? (long long)((unsigned long long)V + (unsigned long long)B) : (long long)((unsigned long long)V - (unsigned long long)B);
            }
            if (postShift) V >>= postShift;
            if (hasPostGain) V = V * (long long)postGain;
        }
        long long acc = V;
        if constexpr (NSEC > 0) {
            // dsp_calc_biquads_int (dsp_biquadSTD.h:34-77).  Four of a section's five products only involve last frame's
            // state: they are issued for ALL sections first (independent chains, wrapping adds commute), so the path through
            // the cascade is one MAC + clamp + shift per section
            long long part[NS_];
#pragma unroll
            for (int k = 0; k < NSEC; k++) part[k] = mac32(sAcc[k], PAR ? xb[k] : xa[k], cf[k][1]);
#pragma unroll
            for (int k = 0; k < NSEC; k++) part[k] = mac32(part[k], PAR ? xa[k] : xb[k], cf[k][2]);
#pragma unroll
            for (int k = 0; k < NSEC; k++) part[k] = mac32(part[k], PAR ? yb[k] : ya[k], cf[k][3]);
#pragma unroll
            for (int k = 0; k < NSEC; k++) part[k] = mac32(part[k], PAR ? ya[k] : yb[k], cf[k][4]);
            int x = q59ToS31(V);                               // the cascade takes X >> 28 (dsp_runtime.c:831)
#pragma unroll
            for (int k = 0; k < NSEC; k++) {
                long long a = mac32(part[k], x, cf[k][0]);
                // checkbiquadsat (dsp_biquadSTD.h:25-32) without a branch: in range <=> -2^27 + 2 <= hi <= 2^27 - 1
                const int hi = hi32(a);
                const long long top = ((long long)(1 << (kMantBQ - 1)) << 32) - 1, bot = -((long long)(1 << (kMantBQ - 1)) << 32);
                a = hi >= (1 << (kMantBQ - 1)) ? top : a;
                a = hi <= 1 - (1 << (kMantBQ - 1)) ? bot : a;
                sAcc[k] = a;
                if (PAR) xa[k] = x; else xb[k] = x;            // the older history word is overwritten: it is next frame's "1"
                x = q59ToS31(a);
                if (PAR) ya[k] = x; else yb[k] = x;
            }
            acc = sAcc[NSEC - 1];
        }
        lastAcc = acc;
        if (exportAcc) { C.blk[accLo + (f & accMask)] = lo32(acc); C.blk[accHi + (f & accMask)] = hi32(acc); }
        if (finKind != FIN_NONE) {
            int v;
            if (finKind == FIN_TRUNC) v = lo32(acc);
            else {
                long long Y = acc;
                if (finHasGain) Y = Y * (long long)finGain;                                        // dsp_runtime.c:636-640
                if (satKind >= SAT_GAIN) { Y >>= kMant; Y = Y * (long long)satGain; }              // :494-534
                if (satKind & 1) Y += tpdfScaledI(C.blk[tpdfOff + (f & tpdfMask)], tpdfShift);     // dspTpdfApply, dsp_tpdf.h:141-145
                v = sat64_031_s32(Y);
            }
            if (dp.staleIdx >= 0 && f == 0) C.st[dp.off + 1 + dp.staleIdx] = v;    // the reference's swap with line[idx0]
            C.blk[postOff + (f & postMask)] = v;
        }
    };
    // Frames alternate parity from the start of the LAUNCH (frame 0 is even), whatever the tile boundaries
    for (int it = 0; it < nIter; it++) {
        __syncthreads();
        const int j = it - 1 - n.depth;
        if (!live || j < 0 || j >= nTiles) continue;
        int f = j * FD;
        const int f1 = min(T, f + FD);                         // FD is even: a tile starts on an even frame
#pragma unroll 1
        for (; f + 1 < f1; f += 2) { frame(f, std::false_type{}); frame(f + 1, std::true_type{}); }
        if (f < f1) frame(f, std::false_type{});                // odd frame count: only the launch's last frame (T odd)
    }
    if (!live) return;
    // back to the reference layout: after an odd number of frames the two history sets have swapped roles
    const bool swapped = (T & 1) != 0;
#pragma unroll
    for (int k = 0; k < NSEC; k++) {
        int* q = C.st + P.pool[n.secStateOff + k];
        q[0] = lo32(sAcc[k]); q[1] = hi32(sAcc[k]);
        q[2] = swapped ? xb[k] : xa[k]; q[3] = swapped ? xa[k] : xb[k]; q[4] = swapped ? yb[k] : ya[k]; q[5] = swapped ? ya[k] : yb[k];
    }
    if (n.a.delayKind == 1) delayWriteBack<1>(da, T, C.st, C.blk + G.aDlyOff[w], nullptr, G.aDlyMask[w]);
    if (n.a.delayKind == 2) delayWriteBack<2>(da, T, C.st, C.blk + G.aDlyOff[w], C.blk + G.aDlyOff[w] + G.aDlyMask[w] + 1, G.aDlyMask[w]);
    if (n.b.delayKind == 1) delayWriteBack<1>(db, T, C.st, C.blk + G.bDlyOff[w], nullptr, G.bDlyMask[w]);
    if (n.b.delayKind == 2) delayWriteBack<2>(db, T, C.st, C.blk + G.bDlyOff[w], C.blk + G.bDlyOff[w] + G.bDlyMask[w] + 1, G.bDlyMask[w]);
    if (n.finKind != FIN_NONE && n.delayN > 0) delayWriteBack<1>(dp, T, C.st, C.blk + postOff, nullptr, postMask);
    if (T > 0) {
        if (n.memOff >= 0) { C.st[n.memOff] = lo32(lastAcc); C.st[n.memOff + 1] = hi32(lastAcc); }       // DSP_STORE_MEM (:760-766)
        for (const DagOperand* o : {&n.a, &n.b})
            if (o->kind == OPD_MUX && o->muxStateOff >= 0) { C.st[o->muxStateOff] = lo32(muxLast); C.st[o->muxStateOff + 1] = hi32(muxLast); }   // :893-896
    }
}

} // namespace

__global__ void __launch_bounds__(kDagMaxThreads, 1)
k_dag(const __grid_constant__ DagPlan P, const Chain2Args A, const __grid_constant__ DagGeom G) {
    extern __shared__ __align__(16) int smem_dag[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp < P.nNodes) {
        switch (P.nodes[warp].nsec) {
        case 0: dagNodeWarp<0>(P, A, G, smem_dag, warp, lane); break;
        case 1: dagNodeWarp<1>(P, A, G, smem_dag, warp, lane); break;
        case 2: dagNodeWarp<2>(P, A, G, smem_dag, warp, lane); break;
        case 3: dagNodeWarp<3>(P, A, G, smem_dag, warp, lane); break;
        case 4: dagNodeWarp<4>(P, A, G, smem_dag, warp, lane); break;
        case 5: dagNodeWarp<5>(P, A, G, smem_dag, warp, lane); break;
        case 6: dagNodeWarp<6>(P, A, G, smem_dag, warp, lane); break;
        case 7: dagNodeWarp<7>(P, A, G, smem_dag, warp, lane); break;
        default: dagNodeWarp<8>(P, A, G, smem_dag, warp, lane); break;
        }
        return;
    }
    const int NS = G.streamsPerCta, T = A.nFrames, W = P.stateWords;
    const int s0 = blockIdx.x * NS, nsHere = min(NS, A.nStreams - s0);
    const int FD = G.tileFrames;
    const int nTiles = (T + FD - 1) / FD, nIter = nTiles + P.maxDepth + 2;
    if (warp == P.nNodes) {
        // ---- input staging (tile `it` at iteration `it`) and the per-stream dither PRNG (lane = stream; DSP_TPDF_CALC,
        // dsp_runtime.c:537-545; dspTpdfCalc, dsp_tpdf.h:103-130)
        const bool own = lane < nsHere;
        const int nIn = P.nIn;
        Prng g = {0, 0, 0, 0}; int tpdfValue = 0, tpdfRandom = 0, dith = 0; bool drew = false;
        int* auxp = nullptr;
        if (own) {
            auxp = A.state + (size_t)(s0 + lane) * W + P.auxOff;
            g.s0 = auxp[AUX_S0]; g.s1 = auxp[AUX_S1]; g.s2 = auxp[AUX_S2]; g.s3 = auxp[AUX_S3];
            tpdfValue = auxp[AUX_TPDF_VALUE]; tpdfRandom = auxp[AUX_TPDF_RANDOM]; dith = auxp[AUX_DITHER];
        }
        const unsigned sbase = (unsigned)__cvta_generic_to_shared(smem_dag);
        // frame of element e of a stream's tile (e = frame * nIn + channel): a small table instead of a division per element
        int* stageFr = smem_dag + G.tabOff + 4 * FD * P.nOut;
        for (int e = lane; e < FD * nIn; e += 32) stageFr[e] = e / nIn;
        __syncwarp();
        for (int it = 0; it < nIter; it++) {
            __syncthreads();
            if (it >= nTiles) continue;
            const int f0 = it * FD, nf = min(FD, T - f0);
            // lane = word inside a stream's interleaved run: consecutive lanes read consecutive words.  Asynchronous copies
            // (LDGSTS): all of the tile's loads are in flight at once instead of one round trip to HBM per stream
            for (int s = 0; s < nsHere; s++) {
                const int* src = A.in + (size_t)(s0 + s) * A.inStreamStride + (size_t)f0 * A.inFrameStride;
                const unsigned blk = sbase + (unsigned)(s * G.perStreamWords + G.rawOff) * 4u;
                for (int e = lane; e < nf * nIn; e += 32) {
                    const int fr = stageFr[e], ch = e - fr * nIn;
                    const unsigned dst = blk + (unsigned)(ch * (G.rawMask + 1) + ((f0 + fr) & G.rawMask)) * 4u;
                    const int* p = src + (size_t)fr * A.inFrameStride + (size_t)ch * A.inChStride;
                    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" :: "r"(dst), "l"(p) : "memory");
                }
            }
            asm volatile("cp.async.commit_group;" ::: "memory");
            // DSP_LOAD_STORE copies (dsp_runtime.c:738-747: no saturation, no STORE mask) leave straight from here:
            // lane = (stream, frame) pair, one pass per copied channel
            if (G.nRawOut) {
                asm volatile("cp.async.wait_all;" ::: "memory");
                __syncwarp();
                for (int k = 0; k < G.nRawOut; k++) {
                    const int ch = G.rawOutCh[k], src = G.rawOutSrc[k];
                    for (int e = lane; e < nsHere * nf; e += 32) {
                        const int s = e / nf, fr = e - s * nf;
                        const int v = src >= 0 ? smem_dag[s * G.perStreamWords + G.rawOff + src * (G.rawMask + 1) + ((f0 + fr) & G.rawMask)] : 0;
                        A.out[(size_t)(s0 + s) * A.outStreamStride + (size_t)(f0 + fr) * A.outFrameStride + (size_t)ch * A.outChStride] = v;
                    }
                }
            }
            if (own) {
                int* row = smem_dag + lane * G.perStreamWords + G.tpdfOff;
                int jf = 0;
                if (P.hasTpdfCalc) {
                    // a table switch on the first frame after a reset: X = 0, no draw, nothing stored (dsp_runtime.c:539-544)
                    if (dith != P.tpdfDither) { dith = P.tpdfDither; row[f0 & G.tpdfMask] = tpdfValue; jf = 1; }
                    if (jf < nf) drew = true;
                    for (; jf < nf; jf++) { tpdfValue = tpdfDraw(g, tpdfRandom); row[(f0 + jf) & G.tpdfMask] = tpdfValue; }
                } else {
                    for (; jf < nf; jf++) row[(f0 + jf) & G.tpdfMask] = tpdfValue;
                }
            }
            asm volatile("cp.async.wait_all;" ::: "memory");       // the tile is in shared memory before the next barrier
        }
        if (auxp) {
            auxp[AUX_S0] = g.s0; auxp[AUX_S1] = g.s1; auxp[AUX_S2] = g.s2; auxp[AUX_S3] = g.s3;
            auxp[AUX_TPDF_VALUE] = tpdfValue; auxp[AUX_TPDF_RANDOM] = tpdfRandom; auxp[AUX_DITHER] = dith;
            if (drew) { int* q = A.state + (size_t)(s0 + lane) * W + P.tpdfDataOff; q[0] = tpdfValue; q[1] = tpdfValue >> 31; }
        }
        return;
    }
    // ---- store warps: tile it - 2 - maxDepth; lane = word inside a stream's output run (interleaved: 128-byte stores).
    // What element e = frame * nOut + channel of a tile reads is the same for every tile and stream: a table built once
    // (row of the channel's node, frame offset behind its DELAY, ring mask, position in the caller's layout)
    const int sw = warp - P.nNodes - 1, nSW = G.nStore;
    const int nOut = P.nOut;
    const int storeMask = ditherMask(P.storeDither);
    int* tabRow = smem_dag + G.tabOff;                  // >= 0: word offset of the post row in a stream's block; -1: reads 0; -2: written elsewhere
    int* tabFr = tabRow + FD * nOut;                     // frame inside the tile minus the delay
    int* tabMask = tabFr + FD * nOut;
    int* tabDst = tabMask + FD * nOut;
    int* tabNode = smem_dag + G.tabOff + 4 * FD * nOut + FD * P.nIn;
    if (sw == 0) {
        for (int e = lane; e < FD * nOut; e += 32) {
            const int fr = e / nOut, ch = e - fr * nOut, node = P.outNode[ch];
            const int dn = (node >= 0 && P.outDelayed[ch]) ? P.nodes[node].delayN : 0;
            tabRow[e] = node >= 0 ? G.postOff[node] : node;
            tabFr[e] = fr - dn;
            tabMask[e] = node >= 0 ? G.postMask[node] : 0;
            tabDst[e] = fr * A.outFrameStride + ch * A.outChStride;
            tabNode[e] = (node >= 0 && dn > 0) ? node : -1;
        }
    }
    for (int it = 0; it < nIter; it++) {
        __syncthreads();
        const int j = it - 2 - P.maxDepth;
        if (j < 0 || j >= nTiles) continue;
        const int f0 = j * FD, nf = min(FD, T - f0);
        for (int s = sw; s < nsHere; s += nSW) {
            const int* blk = smem_dag + s * G.perStreamWords;
            int* dst = A.out + (size_t)(s0 + s) * A.outStreamStride + (size_t)f0 * A.outFrameStride;
#pragma unroll 4
            for (int e = lane; e < nf * nOut; e += 32) {
                const int row = tabRow[e];
                if (row == -2) continue;                           // DSP_LOAD_STORE copy: the staging warp wrote it
                int v = 0;
                if (row >= 0) {
                    const int fd = f0 + tabFr[e];
                    v = blk[row + (fd & tabMask[e])];
                    // a stale ring index: the delayed read of frame 0 returns the old line[n-1] (see DagDelay)
                    if (fd == 0 && tabNode[e] >= 0 && smem_dag[G.staleOff + (tabNode[e] * 32 + s) * 2]) v = smem_dag[G.staleOff + (tabNode[e] * 32 + s) * 2 + 1];
                    v &= storeMask;                                // DSP_STORE masks with the current dither table (:610-633)
                }
                dst[tabDst[e]] = v;
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------ host side
static int pow2AtLeast(int v) { int p = 1; while (p < v) p <<= 1; return p; }

static bool planDagGeometryTile(const DagPlan& P, int nStreams, int numSMs, int FD, DagGeom* geom) {
    DagGeom g{};
    g.tileFrames = FD;
    if (P.nNodes < 1 || P.nNodes > kMaxDagNodes) return false;
    const int maxWarps = kDagMaxThreads / 32;
    if (P.nNodes + 2 > maxWarps) return false;
    g.nStore = std::max(1, std::min(2, maxWarps - P.nNodes - 1));
    g.threads = (P.nNodes + 1 + g.nStore) * 32;
    // every row holds the tile being written plus what its slowest reader still needs.  Writers: staging / dither at
    // iteration `it` write tile it, a node of depth d tile it-1-d; readers: nodes likewise, the store warps tile it-2-maxDepth.
    const int D = P.maxDepth;
    int rawLag = 1, tpdfLag = 1, accLag[kMaxDagNodes];
    for (int w = 0; w < P.nNodes; w++) accLag[w] = 1;
    g.nRawOut = 0;
    for (int ch = 0; ch < P.nOut; ch++) if (P.outNode[ch] == -2) { g.rawOutCh[g.nRawOut] = ch; g.rawOutSrc[g.nRawOut] = P.outRaw[ch]; g.nRawOut++; }
    for (int w = 0; w < P.nNodes; w++) {
        const DagNode& n = P.nodes[w];
        for (const DagOperand* o : {&n.a, &n.b}) {
            if (o->kind == OPD_RAW || o->kind == OPD_MUX) rawLag = std::max(rawLag, 1 + n.depth);
            if (o->kind == OPD_NODE) accLag[o->arg] = std::max(accLag[o->arg], n.depth - P.nodes[o->arg].depth);
        }
        if (n.finKind == FIN_SAT && (n.satKind & 1)) tpdfLag = std::max(tpdfLag, 1 + n.depth);
    }
    int words = 0;
    g.rawMask = pow2AtLeast((rawLag + 1) * FD) - 1;
    g.rawOff = words;  words += std::max(P.nIn, 1) * (g.rawMask + 1);
    g.tpdfMask = pow2AtLeast((tpdfLag + 1) * FD) - 1;
    g.tpdfOff = words; words += g.tpdfMask + 1;
    for (int w = 0; w < P.nNodes; w++) {
        const DagNode& n = P.nodes[w];
        g.accLoOff[w] = g.accHiOff[w] = 0; g.accMask[w] = 0;
        if (n.exportAcc) {
            const int len = pow2AtLeast((accLag[w] + 1) * FD);
            g.accMask[w] = len - 1; g.accLoOff[w] = words; words += len; g.accHiOff[w] = words; words += len;
        }
        g.postOff[w] = 0; g.postMask[w] = 0;
        if (n.finKind != FIN_NONE) {
            const int len = pow2AtLeast((D + 1 - n.depth + 1) * FD + std::max(n.delayN, 0));
            g.postOff[w] = words; g.postMask[w] = len - 1; words += len;
        }
        const DagOperand* ops[2] = {&n.a, &n.b};
        int* offs[2] = {&g.aDlyOff[w], &g.bDlyOff[w]};
        int* masks[2] = {&g.aDlyMask[w], &g.bDlyMask[w]};
        for (int q = 0; q < 2; q++) {
            *offs[q] = 0; *masks[q] = 0;
            if (ops[q]->delayKind && ops[q]->delayN > 0) {
                const int len = pow2AtLeast(ops[q]->delayN + 1);
                *offs[q] = words; *masks[q] = len - 1; words += len * (ops[q]->delayKind == 2 ? 2 : 1);
            }
        }
    }
    g.perStreamWords = words | 1;                                  // odd pitch: lane = stream walks the banks
    // stale-index notes for the store warps + their per-element table (5 words per output element of a tile) + the staging table
    const size_t fixedWords = (size_t)kMaxDagNodes * 32 * 2 + (size_t)FD * (5 * std::max(P.nOut, 1) + std::max(P.nIn, 1));
    int NS = (nStreams + numSMs - 1) / numSMs;
    if (const char* v = getenv("AVDSP_B200_NS_DAG")) { const int e = atoi(v); if (e > 0) NS = e; }
    NS = std::max(1, std::min(NS, 32));
    const size_t budget = (size_t)226 * 1024 / 4 - fixedWords - 8;
    if ((size_t)g.perStreamWords > budget) return false;
    NS = (int)std::min<size_t>((size_t)NS, budget / (size_t)g.perStreamWords);
    g.streamsPerCta = NS;
    g.staleOff = NS * g.perStreamWords;
    g.tabOff = g.staleOff + kMaxDagNodes * 32 * 2;
    g.smemBytes = ((size_t)g.staleOff + fixedWords) * 4;
    *geom = g;
    return true;
}

// 32-frame tiles when a CTA can then hold its share of the streams (one wave), else 16-frame tiles: rows shrink with the tile, and a
// second wave of CTAs costs more than twice as many barriers
bool planDagGeometry(const DagPlan& P, int nStreams, int numSMs, DagGeom* geom) {
    const int want = std::max(1, std::min(32, (nStreams + numSMs - 1) / numSMs));
    DagGeom best{}; bool have = false;
    for (int fd : {32, 16}) {
        DagGeom g{};
        if (!planDagGeometryTile(P, nStreams, numSMs, fd, &g)) continue;
        if (!have || g.streamsPerCta > best.streamsPerCta) { best = g; have = true; }
        if (g.streamsPerCta >= want) break;
    }
    if (have) *geom = best;
    return have;
}

cudaError_t launchDag(const DagPlan& plan, const DagGeom& geom, const Chain2Args& args, cudaStream_t stream) {
    const int blocks = (args.nStreams + geom.streamsPerCta - 1) / geom.streamsPerCta;
    cudaError_t e = cudaFuncSetAttribute(k_dag, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)geom.smemBytes);
    if (e != cudaSuccess) return e;
    k_dag<<<blocks, geom.threads, geom.smemBytes, stream>>>(plan, args, geom);
    return cudaGetLastError();
}

} // namespace avdsp

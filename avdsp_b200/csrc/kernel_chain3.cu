// kernel_chain3.cu -- register-resident cascade executor for the common crossover / EQ program shape
//     LOAD | LOAD_GAIN -> biquad cascade (1..8 sections) -> SAT0DB | SAT0DB_TPDF -> [DELAY] -> STORE(s)
// Fixed point (DSP_FORMAT 2), bit-exact (dsp_calc_biquads_int, runtime/dsp_biquadSTD.h:25-77; dsp_runtime.c:464-491,
// 565-633, 769-794, 827-849).  Programs outside this shape run on k_chain2 (kernel_chain2.cu).
//
// Why a second chain kernel.  k_chain2 gives a lane two sections and links the lanes of a cascade with shuffles; the
// 32x32+64 IMAD.WIDE issues at 1/4 rate and every other ALU instruction next to it costs real time
// (tools/microbench_mix.cu), and k_chain2 spends 13 such instructions per 10 MACs in the section loop plus 36 % of all
// instructions in helper warps that move samples between rings.  Here
//   * a lane owns one cascade -- or one PART of a long cascade, see below -- of one stream: accumulators, histories and
//     coefficients of its sections stay in registers for the whole launch -- no shuffles, no x / accumulator rings.
//     Per section and frame: 5 accumulating IMAD.WIDE + 1 funnel shift + 1 VIADDMNMX (sticky saturation record);
//   * the sections of a lane are SKEWED IN TIME (section k works on frame t-k at step t), so the K section updates of a
//     step are independent chains (an un-skewed cascade is one dependent chain MAC -> shift -> MAC ... per frame and
//     leans on ptxas to interleave the history MACs).  Exact, because section k of frame n only needs section k-1 of
//     the same frame.  The fast loop runs in groups of 6 steps = lcm of the history depths, so the register rotation
//     closes on itself and the loop carries no moves.  The input history of section k+1 is the output history of
//     section k, so a section keeps (acc, y1, y2, y3) only; the reference's separate x1/x2 words are honoured on the
//     first two frames of a launch and rebuilt at its end.  Launch edges (pipeline fill / drain) run a predicated form;
//   * a warp = one chain (or one PART of a chain) x up to 32 streams, so a warp's work is uniform.  One warp issues an
//     IMAD.WIDE every ~6.7 cycles at best, two per sub-partition reach 4.8, three or more ~4.5 (tools/microbench_warps.cu),
//     and a warp that finishes its tile early leaves its neighbour alone with the pipe -- so long cascades are cut into
//     parts of <= 4 sections that run as separate warps (C2: 14 warps of 3 or 4 sections, placed on the sub-partitions
//     by price per frame, placeChain3Warps).  A part hands its output to the next part through a shared-memory row (three
//     tiles deep), one tile later (the consumer part runs F + lag frames behind and waits on a per-part tile counter),
//     so parts never synchronise inside a tile;
//   * the lane reads its input sample straight from the staged PCM tile (cp.async.bulk + mbarrier, issued two tiles
//     ahead by the helper warp; plain copies when the caller's buffer is not 16-byte friendly), applies LOAD_GAIN
//     itself, finishes SAT0DB / SAT0DB_TPDF itself and parks the s.31 value in a shared-memory post ring that doubles
//     as the delay line;
//   * helper warps: warp C runs the per-stream xoshiro128+ (lane = stream) one tile ahead and stages the input; the
//     store warps read the post ring at frame - delay, apply the STORE mask and write 128-byte coalesced runs;
//   * saturation (checkbiquadsat fires on the accumulator's high word): tiles run optimistically and are replayed from
//     a checkpoint (registers for parts of <= 4 sections, shared memory for longer ones) with the exact per-section
//     clamp when the sticky record fired (as in k_chain2).
//
// Ring bookkeeping (F = 32 frames per tile; lag of a warp = its step offset `base` + its sections - 1; gmax = largest lag):
//   row ring  [warp][stream][..] by STEP: the tail of warp w writes at step t the value of frame t - lag_w.  Final parts park the
//             finished s.31 output there (the post ring = the delay line): frame f sits at (f + lag_w) mod R,
//             R >= 2F + gmax + longest delay (power of two); the other parts their last section's y for the next part, in a
//             row of three tiles (slot = tile mod 3: the producer is never more than two tiles ahead of its consumer)
//   tpdf ring [stream][4F]       by frame (the dither warp runs one tile ahead)
//   window i = frames [iF - gmax, (i+1)F - gmax): every chain has finished them when tile i is done.
#include "avdsp_dev.cuh"
#include "kernels.h"
#include <algorithm>
#include <climits>
#include <cstdlib>

namespace avdsp {
namespace {

constexpr int F3 = 32;                  // steps per tile
constexpr int TP3 = 4 * F3 + 1;         // tpdf ring pitch (words)
constexpr int kBarFull3 = 1;            // +parity: inputs of tile i ready and the post ring has room (helpers arrive, cascades wait)
constexpr int kBarDone3 = 3;            // +parity: cascade warps finished tile i (cascades arrive, helpers wait)
#ifndef AVDSP_UNR3
#define AVDSP_UNR3 6
#endif
constexpr unsigned kSatBias3  = (1u << (kMantBQ - 1)) - 2u;     // in range <=> (unsigned)(hi + bias) <= limit
constexpr unsigned kSatLimit3 = (1u << kMantBQ) - 3u;           // (checkbiquadsat, runtime/dsp_biquadSTD.h:25-32)

// named barriers are warp-aligned: reconverge first (lanes take different paths around the per-stream work)
__device__ __forceinline__ void barSync3(int id, int n)   { __syncwarp(); asm volatile("bar.sync %0, %1;" :: "r"(id), "r"(n) : "memory"); }
__device__ __forceinline__ void barArrive3(int id, int n) { __syncwarp(); asm volatile("bar.arrive %0, %1;" :: "r"(id), "r"(n) : "memory"); }
__device__ __forceinline__ unsigned smemAddr3(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ int lds3(unsigned a) { int v; asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(a) : "memory"); return v; }
__device__ __forceinline__ void sts3(unsigned a, int v) { asm volatile("st.shared.b32 [%0], %1;" :: "r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void mbarInit3(unsigned bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbarExpectTx3(unsigned bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tmaLoad3(unsigned dst, const void* src, unsigned bytes, unsigned bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void mbarWait3(unsigned bar, unsigned parity) {
    asm volatile("{\n"
                 ".reg .pred P1;\n"
                 "WAIT3_%=:\n"
                 "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
                 "@P1 bra DONE3_%=;\n"
                 "bra WAIT3_%=;\n"
                 "DONE3_%=:\n"
                 "}" :: "r"(bar), "r"(parity) : "memory");
}

// One cascade in registers, sections skewed in time.  y1/y2/y3[k]: the three most recent outputs of section k (y1 newest);
// section k+1 takes them as its input, x1 and x2.  X1/X2: input history of section 0.  rx1/rx2: the reference's own x1/x2
// words of sections >= 1 as loaded from the state block (they stand in for outputs older than this launch).
template <int NSEC>
struct Casc {
    long long acc[NSEC];
    int y1[NSEC], y2[NSEC], y3[NSEC];
    int X1, X2;
    int rx1[NSEC], rx2[NSEC];
    int b0[NSEC], b1[NSEC], b2[NSEC], a1[NSEC], a2[NSEC];
};

// one step, every section active, OPTIMISTIC: no clamp, only the sticky record of the largest biased high word.
// Returns the accumulator of the last section (frame t - (NSEC-1)).
template <int NSEC>
__device__ __forceinline__ long long cascStep(Casc<NSEC>& L, int xin, unsigned& w0, unsigned& w1) {
    long long acc[NSEC];
    // the NSEC updates are independent: written operand-major so that dependent MACs sit NSEC instructions apart
#pragma unroll
    for (int k = 0; k < NSEC; k++) acc[k] = mac32(L.acc[k], k ? L.y2[k - 1] : L.X1, L.b1[k]);
#pragma unroll
    for (int k = 0; k < NSEC; k++) acc[k] = mac32(acc[k], k ? L.y3[k - 1] : L.X2, L.b2[k]);
#pragma unroll
    for (int k = 0; k < NSEC; k++) acc[k] = mac32(acc[k], L.y1[k], L.a1[k]);
#pragma unroll
    for (int k = 0; k < NSEC; k++) acc[k] = mac32(acc[k], L.y2[k], L.a2[k]);
#pragma unroll
    for (int k = 0; k < NSEC; k++) acc[k] = mac32(acc[k], k ? L.y1[k - 1] : xin, L.b0[k]);
#pragma unroll
    for (int k = 0; k < NSEC; k++) {
        if (k & 1) w1 = max(w1, (unsigned)hi32(acc[k]) + kSatBias3);
        else       w0 = max(w0, (unsigned)hi32(acc[k]) + kSatBias3);
        L.acc[k] = acc[k];
        L.y3[k] = L.y2[k]; L.y2[k] = L.y1[k]; L.y1[k] = q59ToS31(acc[k]);
    }
    L.X2 = L.X1; L.X1 = xin;
    return acc[NSEC - 1];
}
// the same step with the reference's clamp, for any step of the launch: section k commits only when its frame t-k lies in
// [0,T); on the first two frames of a launch the reference's x1/x2 words stand in for outputs older than the launch
template <int NSEC>
__device__ __forceinline__ long long cascStepExact(Casc<NSEC>& L, int xin, int t, int T) {
    int in[NSEC], x1[NSEC], x2[NSEC];
#pragma unroll
    for (int k = 0; k < NSEC; k++) {
        const int f = t - k;
        in[k] = k ? L.y1[k - 1] : xin;
        x1[k] = k ? (f == 0 ? L.rx1[k] : L.y2[k - 1]) : L.X1;
        x2[k] = k ? (f == 0 ? L.rx2[k] : (f == 1 ? L.rx1[k] : L.y3[k - 1])) : L.X2;
    }
    long long last = 0;
#pragma unroll
    for (int k = 0; k < NSEC; k++) {
        if ((unsigned)(t - k) < (unsigned)T) {
            long long acc = L.acc[k];
            acc = mac32(acc, x1[k], L.b1[k]);
            acc = mac32(acc, x2[k], L.b2[k]);
            acc = mac32(acc, L.y1[k], L.a1[k]);
            acc = mac32(acc, L.y2[k], L.a2[k]);
            acc = mac32(acc, in[k], L.b0[k]);
            acc = biquadSat(acc);
            L.acc[k] = acc;
            L.y3[k] = L.y2[k]; L.y2[k] = L.y1[k]; L.y1[k] = q59ToS31(acc);
            if (k == NSEC - 1) last = acc;
        }
    }
    if ((unsigned)t < (unsigned)T) { L.X2 = L.X1; L.X1 = xin; }
    return last;
}

// Unit-gain form (DESIGN.md 4.2a).  A section with b0 = 2^28, b1 + a1 = -2^28, b2 + a2 = 0 (as integers: the 0 dB peaking slots of a
// crossover) satisfies, exactly over the integers and so in Z/2^64,
//     b0 x + b1 x1 + b2 x2 + a1 y1 + a2 y2 = 2^28 (x - x1) + a1 (y1 - x1) + a2 (y2 - x2).
// The part carries z = acc - 2^28 x (x = the section's input of that frame): the 2^28 term telescopes away and
//     z_n = z_{n-1} + a1 d_{n-1} + a2 d_{n-2},   d = y - x = z >> 28,   y_n = x_n + (int)(z_n >> 28)
// (2^28 x has no low bits, so acc >> 28 = x + (z >> 28)): 2 MACs instead of 5, no shift of x, no 33-bit difference.
// That is the reference's arithmetic as long as (a) d fits 32 bits, so that the MAC operand is d itself, and (b) no section saturates,
// so that acc >> 28 is y.  Tiles run optimistically on two sticky records and are replayed exactly when either fires:
//   * hi32(z) in [-2^20, 2^20)  =>  |d| < 2^24;
//   * the part's input x0 in [-(2^31 - 2^27), 2^31 - 2^27].  Section k's input is x0 plus the d of the k sections before it, so every
//     input and output of the part lies within 2^31 - 2^27 + 4 * 2^24 < 2^31 - 32: x + d cannot wrap, and acc >> 28 = y stays inside
//     [-2^31 + 32, 2^31 - 1], the range in which checkbiquadsat (hi32(acc) = (acc >> 28) >> 4 in [-2^27 + 2, 2^27 - 1]) never clamps.
// Both tests are stricter than the reference's clamp: a false alarm costs a replay, never a wrong sample.  A unit section is a
// pass-through plus a rounding residue, so on any but near-full-scale input neither record fires.
constexpr unsigned kUnitZBias = 1u << 20, kUnitZLimit = (1u << 21) - 1u;           // (unsigned)(hi32(z) + bias) <= limit
constexpr unsigned kUnitXBias = 0x78000000u, kUnitXLimit = 2u * 0x78000000u;        // (unsigned)(x0 + bias) <= limit

__device__ __forceinline__ bool unitSection(int b0, int b1, int b2, int a1, int a2) {
    return b0 == (1 << kMantBQ) && (long long)b1 + a1 == -(1ll << kMantBQ) && (long long)b2 + a2 == 0;
}
template <int NSEC>
struct CascU { long long z[NSEC]; int d1[NSEC], d2[NSEC]; };

// one step of a unit-gain part, every section active, optimistic (records only).  Keeps the y / X histories of Casc as they are, so
// that the part leaves the tile in the general layout; returns the accumulator of the last section (frame t - (NSEC-1)).
template <int NSEC>
__device__ __forceinline__ long long unitStep(Casc<NSEC>& L, CascU<NSEC>& U, int xin, unsigned& w0, unsigned& w1, unsigned& wx) {
    long long z[NSEC];
#pragma unroll
    for (int k = 0; k < NSEC; k++) z[k] = mac32(U.z[k], U.d1[k], L.a1[k]);
#pragma unroll
    for (int k = 0; k < NSEC; k++) z[k] = mac32(z[k], U.d2[k], L.a2[k]);
    int y[NSEC];
#pragma unroll
    for (int k = 0; k < NSEC; k++) {
        const int s = q59ToS31(z[k]);
        if (k & 1) w1 = max(w1, (unsigned)hi32(z[k]) + kUnitZBias);
        else       w0 = max(w0, (unsigned)hi32(z[k]) + kUnitZBias);
        y[k] = (k ? L.y1[k - 1] : xin) + s;
        U.z[k] = z[k]; U.d2[k] = U.d1[k]; U.d1[k] = s;
    }
    const int inLast = NSEC > 1 ? L.y1[NSEC - 2] : xin;
    wx = max(wx, (unsigned)xin + kUnitXBias);
#pragma unroll
    for (int k = 0; k < NSEC; k++) { L.y3[k] = L.y2[k]; L.y2[k] = L.y1[k]; L.y1[k] = y[k]; }
    L.X2 = L.X1; L.X1 = xin;
    return z[NSEC - 1] + (long long)((unsigned long long)(long long)inLast << kMantBQ);
}

// SAT0DB_TPDF on the cascade's accumulator (dsp_runtime.c:478-491, dspTpdfApply runtime/dsp_tpdf.h:141-145)
__device__ __forceinline__ int finishTpdf3(long long acc, int tv, bool up, int sh) {
    const long long t = tv;
    acc += up ? (long long)((unsigned long long)t << sh) : (t >> sh);
    return sat64_031_s32(acc);
}

// ------------------------------------------------------------------------------------------------ cascade warps
// MODE bit 0: the source is LOAD_GAIN with gain 1.0 (x = the sample itself); bit 1: SAT0DB_TPDF finish
template <int NSEC, int MODE, bool CKREG>
__device__ __forceinline__ void cascadeWarp(const ChainPlan& P, const Chain2Args& A, const Chain3Geom& G, unsigned char* smem,
                                            int w, int lane) {
    constexpr int LAG = NSEC - 1;
    const int NS = G.streamsPerCta, W = P.h.stateWords, T = A.nFrames;
    const int s0 = blockIdx.x * NS, nsHere = min(NS, A.nStreams - s0);
    const int c = G.warpChain[w];
    const ChainDesc& d = P.chains[c];
    const int sec0 = G.warpFirstSec[w];                     // this warp owns sections [sec0, sec0 + NSEC) of chain c
    const int base = G.warpBase[w];                         // step offset: section k of the warp works on frame t - base - k at step t
    const int LAGA = base + LAG;                            // the warp's tail finishes frame t - LAGA at step t
    const int srcWarp = G.warpSrc[w];                       // -1: the staged PCM tile; else the warp whose row feeds this part
    const bool fin = G.warpFinal[w] != 0;                   // last part of its chain: SAT0DB[_TPDF], delay line, post ring
    const bool live = lane < nsHere;
    // idle lanes (beyond the CTA's streams) shadow the last live stream: they read its rows and load its state, so they compute a
    // copy of it (never garbage that could fire the saturation record and force exact replays of every tile) and store nothing
    const int sl = min(lane, nsHere - 1);
    const int RM = G.postRing - 1;
    const unsigned RM4 = (unsigned)RM << 2, TM4 = (unsigned)(4 * F3 - 1) << 2;
    const unsigned sb = smemAddr3(smem);
    const unsigned postRow = sb + (unsigned)G.warpRowOff[w] + (unsigned)(sl * G.warpPitch[w]) * 4u;
    const unsigned srcRow = sb + (unsigned)G.warpRowOff[max(srcWarp, 0)] + (unsigned)(sl * G.warpPitch[max(srcWarp, 0)]) * 4u;
    volatile int* tileDone = reinterpret_cast<volatile int*>(smem + G.doneOff);       // [warp]: tiles finished
    const unsigned tpdfRow = sb + G.tpdfOff + (unsigned)(sl * TP3) * 4u;
    const unsigned rawRow = sb + G.rawOff + (unsigned)(sl * G.rawPitchBytes) + (unsigned)d.srcCh * 4u;
    const unsigned fb = (unsigned)P.h.nIn * 4u;              // bytes per frame in a staged tile
    const unsigned mbar = sb + G.mbarOff;
    // LOAD: X = the sample, the cascade takes X >> 28; a later part takes the previous part's y as it is (1.0 in Q4.28)
    const int gain = srcWarp >= 0 ? (1 << kMant) : (d.srcKind == SRC_LOAD_GAIN ? d.srcArg : 1);
    const bool tpdfUp = P.h.tpdfShift >= 0;
    const int tpdfSh = (tpdfUp ? P.h.tpdfShift : -P.h.tpdfShift) & 63;
    const bool wantTpdf = fin && (d.satKind & 1) != 0;
    int* st = A.state + (size_t)(s0 + sl) * W;

    Casc<NSEC> L;
    L.X1 = L.X2 = 0;
#pragma unroll
    for (int k = 0; k < NSEC; k++) {
        int cf[5];
        sectionCoefs(P.pool + d.coefOff + 5 * (sec0 + k), A.coefs, A.coefPitch, P.pool[d.coefColOff + sec0 + k], s0 + sl, cf);
        L.b0[k] = cf[0]; L.b1[k] = cf[1]; L.b2[k] = cf[2]; L.a1[k] = cf[3]; L.a2[k] = cf[4];
        L.y3[k] = 0;
        {
            const int* q = st + P.pool[d.secStateOff + sec0 + k];   // [acc_lo, acc_hi, x1, x2, y1, y2] (dsp_biquadSTD.h:45)
            L.acc[k] = (long long)(((unsigned long long)(unsigned)q[1] << 32) | (unsigned)q[0]);
            L.rx1[k] = q[2]; L.rx2[k] = q[3]; L.y1[k] = q[4]; L.y2[k] = q[5];
            if (k == 0) { L.X1 = q[2]; L.X2 = q[3]; }
        }
    }
    // the unit-gain form needs every section of every lane's stream to satisfy the identity (a per-stream coefficient table may
    // break it for some streams: then the whole warp runs the general form).  Parts of 3 and 4 sections only.
    constexpr bool kUnitForm = CKREG && NSEC >= 3;
    bool unit = false;
    if constexpr (kUnitForm) {
        bool ok = true;
#pragma unroll
        for (int k = 0; k < NSEC; k++) ok = ok && unitSection(L.b0[k], L.b1[k], L.b2[k], L.a1[k], L.a2[k]);
        unit = __all_sync(0xffffffffu, ok);
    }
    // delay line (dsp_runtime.c:769-794): ring of n samples, frame f swaps with position (idx0+f) mod n, so the output of frame
    // f is the post value of frame f-n.  The post ring IS the delay line: the n samples the reference ring holds are preloaded
    // as "virtual frames" -n..-1.  A stale index idx0 >= n (delay shortened by reload_params) is used once by the reference
    // and then wraps to 0: frame 0 swaps with ring[idx0], frames >= 1 behave like idx0 = n-1 (same handling as k_chain2).
    const int n = fin ? d.delayN : 0;
    int idx0 = 0, staleIdx = -1;
    if (live && n > 0) {
        const int* ring = st + d.delayOff + 1;
        idx0 = st[d.delayOff];
        const bool stale = idx0 >= n || idx0 < 0;
        for (int k = 0; k < n; k++) {
            const int v = !stale ? ring[(idx0 + k) % n] : (k == 0 ? ring[idx0] : ring[k - 1]);
            sts3(postRow + ((unsigned)((k - n + LAGA) & RM) << 2), v);
        }
        if (stale) { sts3(postRow + ((unsigned)(LAGA & RM) << 2), ring[n - 1]); staleIdx = idx0; idx0 = n - 1; }   // takes the place of post(0)
    }
    const bool anyStale = __any_sync(0xffffffffu, staleIdx >= 0);
    int* ck = reinterpret_cast<int*>(smem + G.ckOff) + (w * 32 + lane);               // [5*maxSec+2 words][cascade threads]
    const int CKP = G.nCascade * 32;
    const int nTiles = (T + G.gmax + F3 - 1) / F3;

    for (int i = 0; i < nTiles; i++) {
        barSync3(kBarFull3 + (i & 1), G.threads);
        const int t0 = i * F3;
        unsigned ra, rstep;                                 // this tile's input: address of step t0, bytes per step
        if (srcWarp < 0) {
            if (G.tma && t0 + F3 <= T) mbarWait3(mbar + 8u * (unsigned)(i & 1), (unsigned)((i >> 1) & 1));
            ra = rawRow + (unsigned)(i & 1) * (unsigned)G.rawStageBytes; rstep = fb;
        } else {
            // the previous part wrote the steps of its tile i-1 into its row: wait until it has finished that tile
            if (i > 0) { while (tileDone[srcWarp] < i) { } __threadfence_block(); __syncwarp(); }
            ra = srcRow + (unsigned)(((i + 2) % 3) * F3) * 4u; rstep = 4u;       // hand-over rows hold three tiles: slot = tile mod 3
        }
        const int tl0 = t0 - base;                          // local step of the tile's first step
        // interior tile: every section of the lane is active on every step, the input tile is complete
        bool exact = !(tl0 >= LAG + 2 && tl0 + F3 <= T && !(anyStale && tl0 <= LAG));
        if (!exact) {
            // checkpoint (registers for short parts, else shared memory: the LSU is idle in this loop), optimistic tile, one
            // vote, rare exact replay
            long long cAcc[CKREG ? NSEC : 1]; int cY1[CKREG ? NSEC : 1], cY2[CKREG ? NSEC : 1], cY3[CKREG ? NSEC : 1], cX1 = 0, cX2 = 0;
            if (CKREG) {
#pragma unroll
                for (int k = 0; k < NSEC; k++) { cAcc[CKREG ? k : 0] = L.acc[k]; cY1[CKREG ? k : 0] = L.y1[k]; cY2[CKREG ? k : 0] = L.y2[k]; cY3[CKREG ? k : 0] = L.y3[k]; }
                cX1 = L.X1; cX2 = L.X2;
            } else {
#pragma unroll
                for (int k = 0; k < NSEC; k++) {
                    ck[(5 * k + 0) * CKP] = lo32(L.acc[k]); ck[(5 * k + 1) * CKP] = hi32(L.acc[k]);
                    ck[(5 * k + 2) * CKP] = L.y1[k]; ck[(5 * k + 3) * CKP] = L.y2[k]; ck[(5 * k + 4) * CKP] = L.y3[k];
                }
                ck[(5 * NSEC) * CKP] = L.X1; ck[(5 * NSEC + 1) * CKP] = L.X2;
            }
            unsigned w0 = 0, w1 = 0, wx = 0;
            unsigned rj = ra;
            unsigned pj = postRow + (fin ? ((unsigned)(t0 & RM) << 2) : (unsigned)((i % 3) * F3) * 4u);
            unsigned tj = (unsigned)((t0 - LAGA) << 2);
            // groups of AVDSP_UNR3 steps: 6 = lcm of the history depths (y1..y3, X1..X2, d1..d2), so the register rotation closes on
            // itself and the loop needs no moves (they would be IMAD.MOVs on the very pipe the MACs saturate); the tile's last steps
            // follow.  step(jj, x) runs one step on input x and returns the value the part writes; jj is a compile-time offset.
            auto runTile = [&](auto&& step) {
                auto one = [&](int jj) {
                    const int smp = lds3(rj); rj += rstep;
                    const int v = step(jj, (MODE & 1) ? smp : q59ToS31(mul32(smp, gain)));
                    if (live) sts3(pj + 4u * jj, v);
                };
                constexpr int kMain = (F3 / AVDSP_UNR3) * AVDSP_UNR3;
#pragma unroll 1
                for (int j0 = 0; j0 < kMain; j0 += AVDSP_UNR3) {
#pragma unroll
                    for (int jj = 0; jj < AVDSP_UNR3; jj++) one(jj);
                    pj += 4u * AVDSP_UNR3; tj += 4u * AVDSP_UNR3;
                }
#pragma unroll
                for (int jj = 0; jj < F3 - kMain; jj++) one(jj);
            };
            bool fired;
            if constexpr (kUnitForm) {
                // unit-gain part: enter the z form from the checkpointed state.  The first step needs d1 = y1 - x1 and d2 = y2 - x2
                // exactly in 32 bits, and the inputs already inside the skewed pipeline within the x0 bound; else this tile runs exact.
                CascU<NSEC> U;
                bool entry = true;
                if (unit) {
#pragma unroll
                    for (int k = 0; k < NSEC; k++) {
                        const int xp1 = k ? L.y2[k - 1] : L.X1, xp2 = k ? L.y3[k - 1] : L.X2;
                        const long long e1 = (long long)L.y1[k] - xp1, e2 = (long long)L.y2[k] - xp2;
                        U.z[k] = L.acc[k] - (long long)((unsigned long long)(long long)xp1 << kMantBQ);
                        U.d1[k] = (int)e1; U.d2[k] = (int)e2;
                        entry = entry && e1 == (long long)(int)e1 && e2 == (long long)(int)e2;
                        if (k < NSEC - 1) entry = entry && (unsigned)L.y1[k] + kUnitXBias <= kUnitXLimit;
                    }
                    entry = __all_sync(0xffffffffu, entry);
                }
                if (unit && !entry) {
                    fired = true;
                } else if (unit) {
                    runTile([&](int jj, int x) {
                        const long long acc = unitStep<NSEC>(L, U, x, w0, w1, wx);
                        if (MODE & 2) return finishTpdf3(acc, lds3(tpdfRow + ((tj + 4u * jj) & TM4)), tpdfUp, tpdfSh);
                        return L.y1[NSEC - 1];
                    });
                    fired = __any_sync(0xffffffffu, max(w0, w1) > kUnitZLimit || wx > kUnitXLimit);
                    if (!fired) {                           // back to the general layout: acc = z + 2^28 * (the section's last input)
#pragma unroll
                        for (int k = 0; k < NSEC; k++)
                            L.acc[k] = U.z[k] + (long long)((unsigned long long)(long long)(k ? L.y2[k - 1] : L.X1) << kMantBQ);
                    }
                }
            }
            if (!kUnitForm || !unit) {
                runTile([&](int jj, int x) {
                    const long long acc = cascStep<NSEC>(L, x, w0, w1);
                    if (MODE & 2) return finishTpdf3(acc, lds3(tpdfRow + ((tj + 4u * jj) & TM4)), tpdfUp, tpdfSh);
                    return q59ToS31(acc);      // SAT0DB of a clamped accumulator is its own >> 28 (replayed exactly if a clamp fired)
                });
                fired = __any_sync(0xffffffffu, max(w0, w1) > kSatLimit3);
            }
            if (fired) {
                if (CKREG) {
#pragma unroll
                    for (int k = 0; k < NSEC; k++) { L.acc[k] = cAcc[CKREG ? k : 0]; L.y1[k] = cY1[CKREG ? k : 0]; L.y2[k] = cY2[CKREG ? k : 0]; L.y3[k] = cY3[CKREG ? k : 0]; }
                    L.X1 = cX1; L.X2 = cX2;
                } else {
#pragma unroll
                    for (int k = 0; k < NSEC; k++) {
                        L.acc[k] = (long long)(((unsigned long long)(unsigned)ck[(5 * k + 1) * CKP] << 32) | (unsigned)ck[(5 * k + 0) * CKP]);
                        L.y1[k] = ck[(5 * k + 2) * CKP]; L.y2[k] = ck[(5 * k + 3) * CKP]; L.y3[k] = ck[(5 * k + 4) * CKP];
                    }
                    L.X1 = ck[(5 * NSEC) * CKP]; L.X2 = ck[(5 * NSEC + 1) * CKP];
                }
                exact = true;
            }
        }
        if (exact) {
            // launch edges (pipeline fill / drain, partial last tile, a stale delay index at frame 0) and replays
#pragma unroll 1
            for (int j = 0; j < F3; j++) {
                const int t = t0 + j, tl = t - base;
                if (tl >= T + LAG) break;
                if (tl < 0) continue;
                const int smp = tl < T ? lds3(ra + (unsigned)j * rstep) : 0;
                const int x = q59ToS31(mul32(smp, gain));
                const long long acc = cascStepExact<NSEC>(L, x, tl, T);
                const int f = tl - LAG;                         // the frame the last section just finished
                if (f >= 0) {
                    int v;
                    if (wantTpdf) v = finishTpdf3(acc, lds3(tpdfRow + ((unsigned)(f << 2) & TM4)), tpdfUp, tpdfSh);
                    else v = q59ToS31(acc);
                    if (live) {
                        if (f == 0 && staleIdx >= 0) st[d.delayOff + 1 + staleIdx] = v;     // the reference's swap with ring[idx0]
                        else sts3(postRow + (fin ? ((unsigned)(t << 2) & RM4) : (unsigned)((i % 3) * F3 + j) * 4u), v);
                    }
                }
            }
        }
        if (!fin) {                                         // the next part may read this tile's steps now
            __syncwarp();
            if (lane == 0) { __threadfence_block(); tileDone[w] = i + 1; }
        }
        barArrive3(kBarDone3 + (i & 1), G.threads);
    }

    if (live) {
        // the pipeline is drained: every section has seen frames 0..T-1.  Back to the reference layout.
#pragma unroll
        for (int k = 0; k < NSEC; k++) {
            int* q = st + P.pool[d.secStateOff + sec0 + k];
            q[0] = lo32(L.acc[k]); q[1] = hi32(L.acc[k]);
            if (k == 0) { q[2] = L.X1; q[3] = L.X2; }
            else if (T >= 2) { q[2] = L.y1[k - 1]; q[3] = L.y2[k - 1]; }
            else if (T == 1) { q[2] = L.y1[k - 1]; q[3] = L.rx1[k]; }
            q[4] = L.y1[k]; q[5] = L.y2[k];
        }
        if (n > 0 && T > 0) {
            // delay line back to the reference's ring layout: frame j sits at position (idx0+j) mod n
            int* ring = st + d.delayOff + 1;
            for (int k = 0; k < n; k++) {
                const long long j = (long long)T - n + k;                    // frames T-n .. T-1 (virtual ones included)
                ring[(int)(((long long)idx0 + j + n) % n)] = lds3(postRow + ((unsigned)(((int)j + LAGA) & RM) << 2));
            }
            st[d.delayOff] = (int)(((long long)idx0 + T) % n);
        }
    }
}

// ------------------------------------------------------------------------------------------------ float class (DSP_FORMAT 3)
// dsp_calc_biquads_float (runtime/dsp_biquadSTD.h:84-119): acc += x*b0; += x1*b1; += x2*b2; += y1*(a1-1); += y2*a2 in THIS order,
// every product truncated (dspMulFloatFloat, dsp_ieee754.h:336-375 == mul.rz.ftz.f32 outside the underflow range, see
// kernel_chain2.cu), every sum rounded to nearest; y = the accumulator itself.  No saturation inside a float cascade, so no
// checkpoint / replay.  Same skew, same rows, same helper warps as the fixed-point form; the lane converts its input sample
// (dspIntToFloatScaled + LOAD_GAIN) and finishes with dspSaturateFloat0db + dsps31Float0DB itself.
template <int NSEC>
struct CascF {
    float acc[NSEC], y1[NSEC], y2[NSEC], y3[NSEC];
    float X1, X2, rx1[NSEC], rx2[NSEC];
    float b0[NSEC], b1[NSEC], b2[NSEC], a1[NSEC], a2[NSEC];
};
__device__ __forceinline__ float maccF3(float acc, float a, float b) { return __fadd_rn(acc, mulFF_fast(a, b)); }

template <int NSEC, bool HUGE = true>
__device__ __forceinline__ float cascStepF(CascF<NSEC>& L, float xin, FltGuard& mn) {
    float acc[NSEC];
#pragma unroll
    for (int k = 0; k < NSEC; k++) acc[k] = maccF3(L.acc[k], k ? L.y1[k - 1] : xin, L.b0[k]);
#pragma unroll
    for (int k = 0; k < NSEC; k++) acc[k] = maccF3(acc[k], k ? L.y2[k - 1] : L.X1, L.b1[k]);
#pragma unroll
    for (int k = 0; k < NSEC; k++) acc[k] = maccF3(acc[k], k ? L.y3[k - 1] : L.X2, L.b2[k]);
#pragma unroll
    for (int k = 0; k < NSEC; k++) acc[k] = maccF3(acc[k], L.y1[k], L.a1[k]);
#pragma unroll
    for (int k = 0; k < NSEC; k++) acc[k] = maccF3(acc[k], L.y2[k], L.a2[k]);
#pragma unroll
    for (int k = 0; k < NSEC; k++) { fltGuard<HUGE>(mn, acc[k]); L.acc[k] = acc[k]; L.y3[k] = L.y2[k]; L.y2[k] = L.y1[k]; L.y1[k] = acc[k]; }
    L.X2 = L.X1; L.X1 = xin;
    return acc[NSEC - 1];
}
// any step of the launch: section k commits only when its frame t-k lies in [0,T); the reference's own x1/x2 words stand in for
// outputs older than the launch on its first two frames
template <int NSEC>
__device__ __forceinline__ float cascStepExactF(CascF<NSEC>& L, float xin, int t, int T, FltGuard& mn) {
    float in[NSEC], x1[NSEC], x2[NSEC];
#pragma unroll
    for (int k = 0; k < NSEC; k++) {
        const int f = t - k;
        in[k] = k ? L.y1[k - 1] : xin;
        x1[k] = k ? (f == 0 ? L.rx1[k] : L.y2[k - 1]) : L.X1;
        x2[k] = k ? (f == 0 ? L.rx2[k] : (f == 1 ? L.rx1[k] : L.y3[k - 1])) : L.X2;
    }
    float last = 0.0f;
#pragma unroll
    for (int k = 0; k < NSEC; k++) {
        if ((unsigned)(t - k) < (unsigned)T) {
            float acc = L.acc[k];
            acc = maccF3(acc, in[k], L.b0[k]);
            acc = maccF3(acc, x1[k], L.b1[k]);
            acc = maccF3(acc, x2[k], L.b2[k]);
            acc = maccF3(acc, L.y1[k], L.a1[k]);
            acc = maccF3(acc, L.y2[k], L.a2[k]);
            fltGuard(mn, acc);
            L.acc[k] = acc;
            L.y3[k] = L.y2[k]; L.y2[k] = L.y1[k]; L.y1[k] = acc;
            if (k == NSEC - 1) last = acc;
        }
    }
    if ((unsigned)t < (unsigned)T) { L.X2 = L.X1; L.X1 = xin; }
    return last;
}

// Interior tiles run two sections per instruction: f32x2 operands (sm_100a FMUL2.FTZ.RZ / FADD2), the same per-element arithmetic
// in half the issue slots.  Pair j holds sections j (low half) and j + NP: the input pair of pair j >= 1 is then the y1 pair of
// pair j-1 as it stands, and its x1/x2 are that pair's y2/y3 -- no half moves between registers except one per step: pair 0
// takes (xin, y1 of section NP-1).  (The first version paired neighbouring sections and spent 0.8 register moves per packed
// multiply on re-pairing, profiles/r2_chain3_c3f_ncu_summary.txt: 45 instructions per step and warp, now 27.)
__device__ __forceinline__ unsigned long long packF3(float lo, float hi) { unsigned long long r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ float loF3(unsigned long long v) { float lo, hi; asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); (void)hi; return lo; }
__device__ __forceinline__ float hiF3(unsigned long long v) { float lo, hi; asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); (void)lo; return hi; }
__device__ __forceinline__ unsigned long long macF3x2(unsigned long long acc, unsigned long long a, unsigned long long b) {
    unsigned long long p;
    asm("mul.rz.ftz.f32x2 %0, %1, %2;" : "=l"(p) : "l"(a), "l"(b));
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(acc) : "l"(acc), "l"(p));
    return acc;
}
template <int NP>
struct CascP { unsigned long long acc[NP], y1[NP], y2[NP], y3[NP], X1, X2, b0[NP], b1[NP], b2[NP], a1[NP], a2[NP]; };
template <int NP, bool HUGE = true>
__device__ __forceinline__ float cascStepP(CascP<NP>& Q, float xin, FltGuard& mn) {
    unsigned long long acc[NP];
    const unsigned long long in0 = packF3(xin, loF3(Q.y1[NP - 1]));     // section NP works on what section NP-1 produced one step ago
#pragma unroll
    for (int j = 0; j < NP; j++) acc[j] = macF3x2(Q.acc[j], j ? Q.y1[j - 1] : in0, Q.b0[j]);
#pragma unroll
    for (int j = 0; j < NP; j++) acc[j] = macF3x2(acc[j], j ? Q.y2[j - 1] : Q.X1, Q.b1[j]);
#pragma unroll
    for (int j = 0; j < NP; j++) acc[j] = macF3x2(acc[j], j ? Q.y3[j - 1] : Q.X2, Q.b2[j]);
#pragma unroll
    for (int j = 0; j < NP; j++) acc[j] = macF3x2(acc[j], Q.y1[j], Q.a1[j]);
#pragma unroll
    for (int j = 0; j < NP; j++) acc[j] = macF3x2(acc[j], Q.y2[j], Q.a2[j]);
#pragma unroll
    for (int j = 0; j < NP; j++) {
        fltGuard<HUGE>(mn, loF3(acc[j])); fltGuard<HUGE>(mn, hiF3(acc[j]));
        Q.acc[j] = acc[j]; Q.y3[j] = Q.y2[j]; Q.y2[j] = Q.y1[j]; Q.y1[j] = acc[j];
    }
    Q.X2 = Q.X1; Q.X1 = in0;
    return hiF3(acc[NP - 1]);
}

// FINM 0: the part hands its float on to the next part; 1: final part, SAT0DB; 2: final part, SAT0DB_TPDF
// SRC 0: the part reads int32 samples from the PCM tile (DSP_FORMAT 3); 1: the previous part's row (floats); 2: float samples
// from the PCM tile (DSP_FORMAT 5: the sample is the float, LOAD_GAIN a plain C multiply)
template <int NSEC, int FINM, int SRC>
__device__ __forceinline__ void cascadeWarpF(const ChainPlan& P, const Chain2Args& A, const Chain3Geom& G, unsigned char* smem, int w, int lane) {
    constexpr int LAG = NSEC - 1;
    constexpr bool fin = FINM != 0;
    constexpr bool PACKED = (NSEC % 2) == 0;
    constexpr int NP = PACKED ? NSEC / 2 : 1;
    const int NS = G.streamsPerCta, W = P.h.stateWords, T = A.nFrames;
    const int s0 = blockIdx.x * NS, nsHere = min(NS, A.nStreams - s0);
    const int c = G.warpChain[w];
    const ChainDesc& d = P.chains[c];
    const int sec0 = G.warpFirstSec[w], base = G.warpBase[w], LAGA = base + LAG, srcWarp = G.warpSrc[w];
    const bool live = lane < nsHere;
    const int sl = min(lane, nsHere - 1);
    const int RM = G.postRing - 1;
    const unsigned RM4 = (unsigned)RM << 2, TM4 = (unsigned)(4 * F3 - 1) << 2;
    const unsigned sb = smemAddr3(smem);
    const unsigned postRow = sb + (unsigned)G.warpRowOff[w] + (unsigned)(sl * G.warpPitch[w]) * 4u;
    const unsigned srcRow = sb + (unsigned)G.warpRowOff[max(srcWarp, 0)] + (unsigned)(sl * G.warpPitch[max(srcWarp, 0)]) * 4u;
    volatile int* tileDone = reinterpret_cast<volatile int*>(smem + G.doneOff);
    const unsigned tpdfRow = sb + G.tpdfOff + (unsigned)(sl * TP3) * 4u;
    const unsigned rawRow = sb + G.rawOff + (unsigned)(sl * G.rawPitchBytes) + (unsigned)d.srcCh * 4u;
    const unsigned fb = (unsigned)P.h.nIn * 4u;
    const unsigned mbar = sb + G.mbarOff;
    constexpr bool FROMPREV = SRC == 1;
    constexpr bool fromPrev = FROMPREV;
    constexpr bool fsmp = SRC == 2;
    const bool hasSrcGain = !fromPrev && d.srcKind == SRC_LOAD_GAIN;
    const float gain = hasSrcGain ? __int_as_float(d.srcArg) : 1.0f;     // mul.rz by 1.0 is exact: LOAD and LOAD_GAIN share the fast form
    const int dither = P.h.storeDither;
    int* st = A.state + (size_t)(s0 + sl) * W;

    CascF<NSEC> L;
    FltGuard mn;            // exactness guard (avdsp_dev.cuh fltGuard): smallest guard word of every value loaded or produced
    bool coefBad = false;   // a table coefficient outside what the guard can bound (fltCoefOutOfRange)
    L.X1 = L.X2 = 0.0f;
#pragma unroll
    for (int k = 0; k < NSEC; k++) {
        int cf[5];
        sectionCoefs(P.pool + d.coefOff + 5 * (sec0 + k), A.coefs, A.coefPitch, P.pool[d.coefColOff + sec0 + k], s0 + sl, cf);
        if (A.coefs) for (int q = 0; q < 5; q++) coefBad |= fltCoefOutOfRange(cf[q]);
        L.b0[k] = __int_as_float(cf[0]); L.b1[k] = __int_as_float(cf[1]); L.b2[k] = __int_as_float(cf[2]);
        L.a1[k] = __int_as_float(cf[3]); L.a2[k] = __int_as_float(cf[4]);
        L.y3[k] = 0.0f;
        const int* q = st + P.pool[d.secStateOff + sec0 + k];       // [acc, -, x1, x2, y1, y2] as floats (dsp_biquadSTD.h:84-119)
        L.acc[k] = __int_as_float(q[0]);
        L.rx1[k] = __int_as_float(q[2]); L.rx2[k] = __int_as_float(q[3]); L.y1[k] = __int_as_float(q[4]); L.y2[k] = __int_as_float(q[5]);
        if (k == 0) { L.X1 = L.rx1[0]; L.X2 = L.rx2[0]; }
        fltGuard(mn, L.acc[k]); fltGuard(mn, L.rx1[k]); fltGuard(mn, L.rx2[k]); fltGuard(mn, L.y1[k]); fltGuard(mn, L.y2[k]);
    }
    if (coefBad) mn.mn = 0u;
    // the post ring is the delay line (ring of s.31 values behind the saturation), exactly as in the fixed-point form
    const int n = fin ? d.delayN : 0;
    int idx0 = 0, staleIdx = -1;
    if (live && n > 0) {
        const int* ring = st + d.delayOff + 1;
        idx0 = st[d.delayOff];
        const bool stale = idx0 >= n || idx0 < 0;
        for (int k = 0; k < n; k++) {
            const int v = !stale ? ring[(idx0 + k) % n] : (k == 0 ? ring[idx0] : ring[k - 1]);
            sts3(postRow + ((unsigned)((k - n + LAGA) & RM) << 2), v);
        }
        if (stale) { sts3(postRow + ((unsigned)(LAGA & RM) << 2), ring[n - 1]); staleIdx = idx0; idx0 = n - 1; }
    }
    const bool anyStale = __any_sync(0xffffffffu, staleIdx >= 0);
    const int nTiles = (T + G.gmax + F3 - 1) / F3;
    // input word -> the cascade's x.  Fast form (the host checked the gains, G.floatFast): hardware convert, exact scale, mul.rz.ftz;
    // no branches -- the previous part's float and the converted sample are both formed, one is selected
    auto sourceFast = [&](int smp) -> float {
        if (fromPrev) return __int_as_float(smp);
        if (fsmp) return __fmul_rn(__int_as_float(smp), gain);     // gain 1.0 for a plain LOAD: exact
        const float x = mulFF_fast(i2f31Fast(smp), gain);
        return smp == 0 ? 0.0f : x;                                // the reference's product of a zero is +0, never -0
    };
    auto sourceExact = [&](int smp) -> float {
        if (fromPrev) return __int_as_float(smp);
        if (fsmp) return __fmul_rn(__int_as_float(smp), gain);
        float x = i2fScaled(smp, 31);
        if (hasSrcGain) { x = mulFF(x, gain); if (smp == 0) x = 0.0f; }
        return x;
    };
    // accumulator -> what goes into the row: the float itself (hand-over) or the finished s.31 sample
    auto emit = [&](float acc, int f) -> int {
        if (FINM == 0) return __float_as_int(acc);
        if (FINM == 2) acc = __fadd_rn(acc, i2fScaled(lds3(tpdfRow + ((unsigned)(f << 2) & TM4)), 31 + dither - 1));
        // the saturated FLOAT goes into the post ring: a DSP_DELAY behind the saturation keeps floats in this format
        // (dspALU_SP_t, dsp_runtime.c:769-794); the store warps convert to s.31 (dsps31Float0DB) like DSP_STORE does
        return __float_as_int(satF(acc));
    };
    // interior tiles park the value BEFORE dspSaturateFloat0db: every reader of the post ring saturates anyway (the store
    // warps' f2s31SatFast is f2s31(satF(.)), the drain below writes satF(.) into the delay line's state words) and satF is idempotent
    auto emitLazy = [&](float acc, int f) -> int {
        if (FINM == 2) acc = __fadd_rn(acc, i2fScaled(lds3(tpdfRow + ((unsigned)(f << 2) & TM4)), 31 + dither - 1));
        return __float_as_int(acc);
    };

    for (int i = 0; i < nTiles; i++) {
        barSync3(kBarFull3 + (i & 1), G.threads);
        const int t0 = i * F3;
        unsigned ra, rstep;
        if (!FROMPREV) {
            if (G.tma && t0 + F3 <= T) mbarWait3(mbar + 8u * (unsigned)(i & 1), (unsigned)((i >> 1) & 1));
            ra = rawRow + (unsigned)(i & 1) * (unsigned)G.rawStageBytes; rstep = fb;
        } else {
            if (i > 0) { while (tileDone[srcWarp] < i) { } __threadfence_block(); __syncwarp(); }
            ra = srcRow + (unsigned)(((i + 2) % 3) * F3) * 4u; rstep = 4u;
        }
        const int tl0 = t0 - base;
        const bool interior = G.floatFast && tl0 >= LAG + 2 && tl0 + F3 <= T && !(anyStale && tl0 <= LAG);
        if (interior) {
            unsigned rj = ra;
            unsigned pj = postRow + (fin ? ((unsigned)(t0 & RM) << 2) : (unsigned)((i % 3) * F3) * 4u);
            int fj = t0 - LAGA;
            CascP<NP> Q;
            if constexpr (PACKED) {
                Q.X1 = packF3(L.X1, L.y2[NP - 1]); Q.X2 = packF3(L.X2, L.y3[NP - 1]);
#pragma unroll
                for (int j = 0; j < NP; j++) {
                    const int e = j, o = j + NP;
                    Q.acc[j] = packF3(L.acc[e], L.acc[o]);
                    Q.y1[j] = packF3(L.y1[e], L.y1[o]); Q.y2[j] = packF3(L.y2[e], L.y2[o]); Q.y3[j] = packF3(L.y3[e], L.y3[o]);
                    Q.b0[j] = packF3(L.b0[e], L.b0[o]); Q.b1[j] = packF3(L.b1[e], L.b1[o]); Q.b2[j] = packF3(L.b2[e], L.b2[o]);
                    Q.a1[j] = packF3(L.a1[e], L.a1[o]); Q.a2[j] = packF3(L.a2[e], L.a2[o]);
                }
            }
            auto step = [&](int jj) {
                const int smp = lds3(rj); rj += rstep;
                float acc;
                const float xs_ = sourceFast(smp);
                if (!FROMPREV) fltGuard(mn, xs_);
                // (the huge side of the guard on every sixth step: avdsp_dev.cuh; jj is a constant after unrolling)
                if constexpr (PACKED) acc = (jj % 6 == 0) ? cascStepP<NP, true>(Q, xs_, mn) : cascStepP<NP, false>(Q, xs_, mn);
                else acc = (jj % 6 == 0) ? cascStepF<NSEC, true>(L, xs_, mn) : cascStepF<NSEC, false>(L, xs_, mn);
                const int v = emitLazy(acc, fj + jj);
                if (live) sts3(pj + 4u * jj, v);
            };
            constexpr int kMain = (F3 / AVDSP_UNR3) * AVDSP_UNR3;
#pragma unroll 1
            for (int j0 = 0; j0 < kMain; j0 += AVDSP_UNR3) {
#pragma unroll
                for (int jj = 0; jj < AVDSP_UNR3; jj++) step(jj);
                pj += 4u * AVDSP_UNR3; fj += AVDSP_UNR3;
            }
#pragma unroll
            for (int jj = 0; jj < F3 - kMain; jj++) step(jj);
            if constexpr (PACKED) {
                L.X1 = loF3(Q.X1); L.X2 = loF3(Q.X2);
#pragma unroll
                for (int j = 0; j < NP; j++) {
                    const int e = j, o = j + NP;
                    L.acc[e] = loF3(Q.acc[j]); L.acc[o] = hiF3(Q.acc[j]);
                    L.y1[e] = loF3(Q.y1[j]); L.y1[o] = hiF3(Q.y1[j]); L.y2[e] = loF3(Q.y2[j]); L.y2[o] = hiF3(Q.y2[j]);
                    L.y3[e] = loF3(Q.y3[j]); L.y3[o] = hiF3(Q.y3[j]);
                }
            }
        } else {
#pragma unroll 1
            for (int j = 0; j < F3; j++) {
                const int t = t0 + j, tl = t - base;
                if (tl >= T + LAG) break;
                if (tl < 0) continue;
                const int smp = tl < T ? lds3(ra + (unsigned)j * rstep) : 0;
                const float xs_ = G.floatFast ? sourceFast(smp) : sourceExact(smp);
                if (!FROMPREV && tl < T) fltGuard(mn, xs_);
                const float acc = cascStepExactF<NSEC>(L, xs_, tl, T, mn);
                const int f = tl - LAG;
                if (f >= 0) {
                    const int v = emit(acc, f);
                    if (live) {
                        if (f == 0 && staleIdx >= 0) st[d.delayOff + 1 + staleIdx] = v;
                        else sts3(postRow + (fin ? ((unsigned)(t << 2) & RM4) : (unsigned)((i % 3) * F3 + j) * 4u), v);
                    }
                }
            }
        }
        if (!fin) {
            __syncwarp();
            if (lane == 0) { __threadfence_block(); tileDone[w] = i + 1; }
        }
        barArrive3(kBarDone3 + (i & 1), G.threads);
    }
    if (live) {
#pragma unroll
        for (int k = 0; k < NSEC; k++) {
            int* q = st + P.pool[d.secStateOff + sec0 + k];
            q[0] = __float_as_int(L.acc[k]);
            if (k == 0) { q[2] = __float_as_int(L.X1); q[3] = __float_as_int(L.X2); }
            else if (T >= 2) { q[2] = __float_as_int(L.y1[k - 1]); q[3] = __float_as_int(L.y2[k - 1]); }
            else if (T == 1) { q[2] = __float_as_int(L.y1[k - 1]); q[3] = __float_as_int(L.rx1[k]); }
            q[4] = __float_as_int(L.y1[k]); q[5] = __float_as_int(L.y2[k]);
        }
        if (fltGuardFired(mn) && A.redo) A.redo[s0 + sl] = 1;
        if (n > 0 && T > 0) {
            int* ring = st + d.delayOff + 1;
            for (int k = 0; k < n; k++) {
                const long long j = (long long)T - n + k;
                ring[(int)(((long long)idx0 + j + n) % n)] = __float_as_int(satF(__int_as_float(lds3(postRow + ((unsigned)(((int)j + LAGA) & RM) << 2)))));
            }
            st[d.delayOff] = (int)(((long long)idx0 + T) % n);
        }
    }
}
template <int NSEC>
__device__ __forceinline__ void cascadeWarpFin(const ChainPlan& P, const Chain2Args& A, const Chain3Geom& G, unsigned char* smem, int w, int lane) {
    const int finm = !G.warpFinal[w] ? 0 : (P.chains[G.warpChain[w]].satKind & 1) ? 2 : 1;
    const int src = G.warpSrc[w] >= 0 ? 1 : (P.h.sampleInt ? 0 : 2);
    switch (finm * 3 + src) {
    case 0:  cascadeWarpF<NSEC, 0, 0>(P, A, G, smem, w, lane); break;
    case 1:  cascadeWarpF<NSEC, 0, 1>(P, A, G, smem, w, lane); break;
    case 2:  cascadeWarpF<NSEC, 0, 2>(P, A, G, smem, w, lane); break;
    case 3:  cascadeWarpF<NSEC, 1, 0>(P, A, G, smem, w, lane); break;
    case 4:  cascadeWarpF<NSEC, 1, 1>(P, A, G, smem, w, lane); break;
    case 5:  cascadeWarpF<NSEC, 1, 2>(P, A, G, smem, w, lane); break;
    case 6:  cascadeWarpF<NSEC, 2, 0>(P, A, G, smem, w, lane); break;
    case 7:  cascadeWarpF<NSEC, 2, 1>(P, A, G, smem, w, lane); break;
    default: cascadeWarpF<NSEC, 2, 2>(P, A, G, smem, w, lane); break;
    }
}

template <int NSEC, bool CKREG>
__device__ __forceinline__ void cascadeWarpMode(const ChainPlan& P, const Chain2Args& A, const Chain3Geom& G, unsigned char* smem,
                                                int w, int lane, int mode) {
    switch (mode) {
    case 0:  cascadeWarp<NSEC, 0, CKREG>(P, A, G, smem, w, lane); break;
    case 1:  cascadeWarp<NSEC, 1, CKREG>(P, A, G, smem, w, lane); break;
    case 2:  cascadeWarp<NSEC, 2, CKREG>(P, A, G, smem, w, lane); break;
    default: cascadeWarp<NSEC, 3, CKREG>(P, A, G, smem, w, lane); break;
    }
}

// store pass of one stream's window, interleaved output with NOUT (power of two) channels: 32/NOUT frames per pass, one
// 128-byte run per pass; per-lane constants (row, lag - delay, mask) in registers
// post-ring word -> s.31 sample: the fixed-point form parks it as such, the float form parks the saturated float
template <bool FLT, bool FSMP> __device__ __forceinline__ int post3(int v) {
    if (FLT) return FSMP ? __float_as_int(satF(__int_as_float(v))) : f2s31SatFast(v);       // DSP_FORMAT 5 stores the float itself
    return v;
}

template <int NOUT, bool FLT, bool FSMP>
__device__ __forceinline__ void storeTile3(int* __restrict__ out, unsigned rowA, unsigned p4, unsigned RM4, int mask, bool clean,
                                           int f0, int fs, int T) {
    constexpr int FPP = 32 / NOUT, NPASS = F3 / FPP;
    if (clean) {
#pragma unroll
        for (int p = 0; p < NPASS; p++) out[p * 32] = post3<FLT, FSMP>(lds3(rowA + ((p4 + (unsigned)(p * FPP * 4)) & RM4))) & mask;
    } else {
#pragma unroll 1
        for (int p = 0; p < NPASS; p++) {
            const int f = f0 + p * FPP + fs;
            if (f >= 0 && f < T) out[p * 32] = post3<FLT, FSMP>(lds3(rowA + ((p4 + (unsigned)(p * FPP * 4)) & RM4))) & mask;
        }
    }
}

// all streams of one store warp for one window: the channel-count dispatch sits outside the stream loop, the loop itself is
// pointer bumps + the passes
template <int NOUT, bool FLT, bool FSMP>
__device__ __forceinline__ void storeStreams3(int* __restrict__ out, size_t outStep, unsigned rowA, unsigned rowStep, int cnt, unsigned p4,
                                              unsigned RM4, int mask, bool clean, int f0, int fs, int T) {
#pragma unroll 1
    for (int s = 0; s < cnt; s++, out += outStep, rowA += rowStep) storeTile3<NOUT, FLT, FSMP>(out, rowA, p4, RM4, mask, clean, f0, fs, T);
}

} // namespace

// MAXSEC = 8: whole cascades, up to 12 warps of 168 registers;  MAXSEC = 4: cascades cut into parts, up to 16 warps of 128
// FLT: the float class (DSP_FORMAT 3) as its own instance, so that the fixed-point kernel's code (instruction-cache sensitive) is unchanged
template <int MAXSEC, bool FLT = false>
__global__ void __launch_bounds__(MAXSEC > 4 ? kChain3MaxThreads : kChain3MaxThreadsParts, 1)
k_chain3(const __grid_constant__ ChainPlan P, const Chain2Args A, const __grid_constant__ Chain3Geom G) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31;
    const int role = G.warpRole[threadIdx.x >> 5];          // >= 0: cascade warp (index); -1: dither warp; <= -2: store warp -2-k
    if constexpr (FLT) {
        if (role >= 0) {
            switch (G.warpNsec[role]) {
            case 1: cascadeWarpFin<1>(P, A, G, smem_raw, role, lane); break;
            case 2: cascadeWarpFin<2>(P, A, G, smem_raw, role, lane); break;
            case 3: cascadeWarpFin<3>(P, A, G, smem_raw, role, lane); break;
            default: cascadeWarpFin<4>(P, A, G, smem_raw, role, lane); break;
            }
            return;
        }
    } else if (role >= 0) {
        const int warp = role;
        const ChainDesc& d = P.chains[G.warpChain[warp]];
        const bool unity = G.warpSrc[warp] >= 0 || (d.srcKind == SRC_LOAD_GAIN && d.srcArg == (1 << kMant));
        const int mode = (unity ? 1 : 0) | ((G.warpFinal[warp] && (d.satKind & 1)) ? 2 : 0);
        switch (G.warpNsec[warp]) {
        case 1: cascadeWarpMode<1, (MAXSEC <= 4)>(P, A, G, smem_raw, warp, lane, mode); break;
        case 2: cascadeWarpMode<2, (MAXSEC <= 4)>(P, A, G, smem_raw, warp, lane, mode); break;
        case 3: cascadeWarpMode<3, (MAXSEC <= 4)>(P, A, G, smem_raw, warp, lane, mode); break;
        case 4: cascadeWarpMode<4, (MAXSEC <= 4)>(P, A, G, smem_raw, warp, lane, mode); break;
        default:
            if constexpr (MAXSEC > 4) {
                switch (G.warpNsec[warp]) {
                case 5: cascadeWarpMode<5, (MAXSEC <= 4)>(P, A, G, smem_raw, warp, lane, mode); break;
                case 6: cascadeWarpMode<6, (MAXSEC <= 4)>(P, A, G, smem_raw, warp, lane, mode); break;
                case 7: cascadeWarpMode<7, (MAXSEC <= 4)>(P, A, G, smem_raw, warp, lane, mode); break;
                default: cascadeWarpMode<8, (MAXSEC <= 4)>(P, A, G, smem_raw, warp, lane, mode); break;
                }
            }
            break;
        }
        return;
    }
    // =============================================================================== helper warps
    const int NS = G.streamsPerCta, W = P.h.stateWords, T = A.nFrames;
    const int s0 = blockIdx.x * NS, nsHere = min(NS, A.nStreams - s0);
    const int gmax = G.gmax;
    const int nTiles = (T + gmax + F3 - 1) / F3;
    const int hw = -role - 1;                               // 0: dither PRNG + input staging; 1..nStore: store warps
    const unsigned sb = smemAddr3(smem_raw);
    const unsigned RM4 = (unsigned)(G.postRing - 1) << 2;

    if (hw == 0) {
        // ---- per-stream dither PRNG (lane = stream; DSP_TPDF_CALC, dsp_runtime.c:537-545) one tile ahead of the cascades, and
        // the input tiles: bulk copies two tiles ahead, or plain copies one tile ahead where the bulk copy cannot be used
        const bool own = lane < nsHere;
        const bool hasCalc = P.h.hasTpdfCalc != 0;
        const int nIn = P.h.nIn;
        Prng g = {0, 0, 0, 0}; int tpdfValue = 0, tpdfRandom = 0, dith = 0; bool drew = false;
        int* auxp = nullptr;
        if (own) {
            auxp = A.state + (size_t)(s0 + lane) * W + P.h.auxOff;
            g.s0 = auxp[AUX_S0]; g.s1 = auxp[AUX_S1]; g.s2 = auxp[AUX_S2]; g.s3 = auxp[AUX_S3];
            tpdfValue = auxp[AUX_TPDF_VALUE]; tpdfRandom = auxp[AUX_TPDF_RANDOM]; dith = auxp[AUX_DITHER];
        }
        const unsigned mbar = sb + G.mbarOff;
        const unsigned rowBytes = (unsigned)(F3 * nIn * 4);
        if (G.tma && lane == 0) { mbarInit3(mbar, 1); mbarInit3(mbar + 8, 1); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
        if (lane < kChain3MaxWarps) reinterpret_cast<volatile int*>(smem_raw + G.doneOff)[lane] = 0;     // per-part tile counters
        __syncwarp();
        auto issueTile = [&](int it) {                      // full tiles by TMA
            if (!G.tma || (it + 1) * F3 > T) return;
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            const unsigned bar = mbar + 8u * (unsigned)(it & 1);
            if (lane == 0) mbarExpectTx3(bar, (unsigned)nsHere * rowBytes);
            __syncwarp();
            if (own) {
                const int* src = A.in + (size_t)(s0 + lane) * A.inStreamStride + (size_t)(it * F3) * A.inFrameStride;
                tmaLoad3(sb + G.rawOff + (unsigned)(it & 1) * (unsigned)G.rawStageBytes + (unsigned)(lane * G.rawPitchBytes), src, rowBytes, bar);
            }
        };
        auto copyTile = [&](int it) {                       // everything else (partial last tile, planar or unaligned buffers)
            const int f0 = it * F3;
            if (f0 >= T || (G.tma && f0 + F3 <= T)) return;
            const int nf = min(F3, T - f0);
            const unsigned dst0 = sb + G.rawOff + (unsigned)(it & 1) * (unsigned)G.rawStageBytes;
            // lane = channel-sample inside a stream's row: consecutive lanes read consecutive words of interleaved PCM
            for (int s = 0; s < nsHere; s++) {
                const int* src = A.in + (size_t)(s0 + s) * A.inStreamStride + (size_t)f0 * A.inFrameStride;
                for (int e = lane; e < nf * nIn; e += 32) {
                    const int fr = e / nIn, ch = e - fr * nIn;
                    sts3(dst0 + (unsigned)(s * G.rawPitchBytes) + 4u * (unsigned)e, src[(size_t)fr * A.inFrameStride + (size_t)ch * A.inChStride]);
                }
            }
        };
        auto ditherTile = [&](int it) {
            const int f0 = it * F3;
            if (f0 >= T || !own) return;
            const unsigned row = sb + G.tpdfOff + (unsigned)(lane * TP3 + (it & 3) * F3) * 4u;
            const int nf = min(F3, T - f0);
            int j = 0;
            if (hasCalc) {
                // a table switch on the first frame after a reset: no draw (dsp_runtime.c:539-544)
                if (dith != P.h.tpdfDither) { dith = P.h.tpdfDither; sts3(row, tpdfValue); j = 1; }
                if (j < nf) drew = true;
                for (; j < nf; j++) { tpdfValue = tpdfDraw(g, tpdfRandom); sts3(row + 4u * j, tpdfValue); }
            } else {
                for (; j < nf; j++) sts3(row + 4u * j, tpdfValue);
            }
        };
        issueTile(0);
        issueTile(1);
        copyTile(0);
        ditherTile(0);
        barArrive3(kBarFull3 + 0, G.threads);
        for (int i = 0; i < nTiles; i++) {
            if (i + 1 < nTiles) { copyTile(i + 1); ditherTile(i + 1); barArrive3(kBarFull3 + ((i + 1) & 1), G.threads); }
            barSync3(kBarDone3 + (i & 1), G.threads);
            issueTile(i + 2);                               // the cascades are done with this parity's buffer
        }
        if (auxp) {
            auxp[AUX_S0] = g.s0; auxp[AUX_S1] = g.s1; auxp[AUX_S2] = g.s2; auxp[AUX_S3] = g.s3;
            auxp[AUX_TPDF_VALUE] = tpdfValue; auxp[AUX_TPDF_RANDOM] = tpdfRandom; auxp[AUX_DITHER] = dith;
            if (drew) {   // TPDF_CALC leaves its last value (as an ALU word) in the data area (dsp_runtime.c:541-543)
                int* q = A.state + (size_t)(s0 + lane) * W + P.h.tpdfDataOff;
                if (FLT) q[0] = __float_as_int(i2fScaled(tpdfValue, 31));          // the ALU word is a float in DSP_FORMAT 3
                else { q[0] = tpdfValue; q[1] = tpdfValue >> 31; }
            }
        }
        return;
    }

    // ---- store warps: post ring at (frame + lag - delay) -> STORE mask -> global
    const int sw = hw - 1, nSW = G.nStore;
    const int nOut = P.h.nOut;
    const bool fsmp = FLT && !P.h.sampleInt;                 // DSP_FORMAT 5: floats out, no STORE mask
    const int storeMask = fsmp ? -1 : ditherMask(P.h.storeDither);
    const bool laneOut = A.outChStride == 1 && A.outFrameStride == nOut;      // interleaved: lane = (frame inside a pass, channel)
    const int bCh = lane % nOut, bFs = lane / nOut;
    const int bChain = P.h.chainOfOut[bCh];
    const unsigned bRow = bChain >= 0 ? (unsigned)G.warpRowOff[G.chainRow[bChain]] : (unsigned)G.warpRowOff[G.chainRow[0]];
    const int bOff = bChain >= 0 ? G.chainLag[bChain] - P.chains[bChain].delayN : 0;
    const int bMask = bChain >= 0 ? storeMask : 0;          // outputs no path writes read as 0
    barArrive3(kBarFull3 + 0, G.threads);
    for (int i = 0; i < nTiles; i++) {
        if (i + 1 < nTiles) barArrive3(kBarFull3 + ((i + 1) & 1), G.threads);     // window i-1 is stored: its ring span may be reused
        barSync3(kBarDone3 + (i & 1), G.threads);
        const int f0 = i * F3 - gmax;                       // window i
        const bool clean = f0 >= 0 && f0 + F3 <= T;
        if (laneOut) {
            const unsigned p4 = (unsigned)((f0 + bFs + bOff) << 2);
            const int cnt = nsHere > sw ? (nsHere - sw + nSW - 1) / nSW : 0;
            int* out = A.out + (size_t)(s0 + sw) * A.outStreamStride + (long long)f0 * A.outFrameStride + lane;
            const size_t outStep = (size_t)nSW * (size_t)A.outStreamStride;
            const unsigned rowA = sb + bRow + (unsigned)(sw * G.postPitch) * 4u, rowStep = (unsigned)(nSW * G.postPitch) * 4u;
            if (FLT && fsmp) {
                switch (nOut) {
                case 1:  storeStreams3<1, FLT, true>(out, outStep, rowA, rowStep, cnt, p4, RM4, bMask, clean, f0, bFs, T); break;
                case 2:  storeStreams3<2, FLT, true>(out, outStep, rowA, rowStep, cnt, p4, RM4, bMask, clean, f0, bFs, T); break;
                case 4:  storeStreams3<4, FLT, true>(out, outStep, rowA, rowStep, cnt, p4, RM4, bMask, clean, f0, bFs, T); break;
                case 8:  storeStreams3<8, FLT, true>(out, outStep, rowA, rowStep, cnt, p4, RM4, bMask, clean, f0, bFs, T); break;
                case 16: storeStreams3<16, FLT, true>(out, outStep, rowA, rowStep, cnt, p4, RM4, bMask, clean, f0, bFs, T); break;
                default: storeStreams3<32, FLT, true>(out, outStep, rowA, rowStep, cnt, p4, RM4, bMask, clean, f0, bFs, T); break;
                }
            } else {
                switch (nOut) {
                case 1:  storeStreams3<1, FLT, false>(out, outStep, rowA, rowStep, cnt, p4, RM4, bMask, clean, f0, bFs, T); break;
                case 2:  storeStreams3<2, FLT, false>(out, outStep, rowA, rowStep, cnt, p4, RM4, bMask, clean, f0, bFs, T); break;
                case 4:  storeStreams3<4, FLT, false>(out, outStep, rowA, rowStep, cnt, p4, RM4, bMask, clean, f0, bFs, T); break;
                case 8:  storeStreams3<8, FLT, false>(out, outStep, rowA, rowStep, cnt, p4, RM4, bMask, clean, f0, bFs, T); break;
                case 16: storeStreams3<16, FLT, false>(out, outStep, rowA, rowStep, cnt, p4, RM4, bMask, clean, f0, bFs, T); break;
                default: storeStreams3<32, FLT, false>(out, outStep, rowA, rowStep, cnt, p4, RM4, bMask, clean, f0, bFs, T); break;
                }
            }
        } else {
            // any other layout (planar): lane = frame, channels in a loop; consecutive lanes store consecutive frames
            const int f = f0 + lane;
            if (f >= 0 && f < T)
                for (int sl = sw; sl < nsHere; sl += nSW)
                    for (int ch = 0; ch < nOut; ch++) {
                        const int oc = P.h.chainOfOut[ch];
                        int v = 0;
                        if (oc >= 0) {
                            const int off = G.chainLag[oc] - P.chains[oc].delayN;
                            { const int wv_ = lds3(sb + (unsigned)G.warpRowOff[G.chainRow[oc]] + (unsigned)(sl * G.postPitch) * 4u + ((unsigned)((f + off) << 2) & RM4)); v = (fsmp ? post3<FLT, true>(wv_) : post3<FLT, false>(wv_)) & storeMask; }
                        }
                        A.out[(size_t)(s0 + sl) * A.outStreamStride + (size_t)f * A.outFrameStride + (size_t)ch * A.outChStride] = v;
                    }
        }
    }
}

// ------------------------------------------------------------------------------------------------ host side
static int envInt3(const char* name, int dflt) { const char* v = getenv(name); return (v && *v) ? atoi(v) : dflt; }

bool chain3Supports(const ChainPlan& plan) {
    const ChainHeader& h = plan.h;
    if (h.aluClass != ALU_INT64 && h.aluClass != ALU_F32) return false;                        // DSP_FORMAT 2, 3 and 5
    if (h.aluClass == ALU_F32 && !chainFloatCoefsInRange(plan)) return false;
    if (h.nChains <= 0 || h.nChains > kChain3MaxChains || h.nIn <= 0) return false;
    if (h.nOut <= 0 || h.nOut > 32 || (h.nOut & (h.nOut - 1)) != 0) return false;
    if (h.nRaw || h.nDelayFirst || h.nMemCopy) return false;
    for (int c = 0; c < h.nChains; c++) {
        const ChainDesc& d = plan.chains[c];
        if (d.nsec < 1 || d.nsec > 16) return false;        // up to four parts of four sections (plain finish), see planChain3Geometry
        if (d.srcKind != SRC_LOAD && d.srcKind != SRC_LOAD_GAIN) return false;
        if (d.srcCh < 0 || d.srcCh >= h.nIn) return false;
        if (d.hasGain || d.delayFirst) return false;
        if (d.satKind != SAT_PLAIN && d.satKind != SAT_TPDF) return false;
        if (d.delayN < 0) return false;
    }
    return true;
}

// What one warp costs per frame on its sub-partition: IMAD.WIDE on the MAC pipe (the planned form, and the general form a CTA
// falls back to when a per-stream coefficient row breaks the unit-gain identity), and the rest in issue cycles beside them.
// Item k < nCascade is cascade warp k; then the dither warp, then the store warps.  A section issues a shift and a saturation
// record beside its MACs (unit-gain form: one add more), a part 4 instructions of bookkeeping.  The TPDF finish, the source
// gain and the helper warps are priced from tools/chain3_placement_sweep.py (profiles/r7_chain3_placement_sweep.jsonl): on
// the tile barrier's critical path they cost more than their instruction counts, and these prices rank the timed C2, C3 and
// C3-float placements (Spearman 0.92-0.98 against the measured times).
struct Chain3Price { int macs, other, macsGeneral, otherGeneral; };

static Chain3Price chain3Price(const ChainPlan& plan, const Chain3Geom& g, int k) {
    if (k == g.nCascade) return {0, 20, 0, 20};
    if (k > g.nCascade) {                                    // 4 cycles per 32 output words, shared by the store warps
        const int words = plan.h.nOut * g.streamsPerCta;
        const int o = (4 * words + 16 * g.nStore) / (32 * g.nStore);
        return {0, o, 0, o};
    }
    const ChainDesc& d = plan.chains[g.warpChain[k]];
    const int n = g.warpNsec[k];
    int extra = 4;
    if (g.warpFinal[k] && (d.satKind & 1)) extra += 30;
    if (g.warpSrc[k] < 0 && !(d.srcKind == SRC_LOAD_GAIN && d.srcArg == (1 << kMant))) extra += 24;
    return {(g.warpUnit[k] ? 2 : 5) * n, (g.warpUnit[k] ? 3 : 2) * n + extra, 5 * n, 2 * n + extra};
}

// Price of a sub-partition per frame in issue cycles: the MAC pipe takes about 4 cycles per IMAD.WIDE (tools/microbench_warps.cu:
// 4.05 at best), the other instructions are added on top (they share the issue slots and the tile barrier waits for all of them)
static int chain3BinCost(int macs, int other) { return 4 * macs + other; }

std::string chain3PlacementTrace(const ChainPlan& plan, const Chain3Geom& g) {
    const int total = g.threads / 32;
    int itemOf[32];                                          // hardware warp id -> item
    for (int id = 0; id < total; id++) itemOf[id] = g.warpRole[id] >= 0 ? g.warpRole[id] : g.nCascade - 1 - g.warpRole[id];
    int bin[32];
    for (int id = 0; id < total; id++) bin[itemOf[id]] = id & 3;
    std::string s = "chain kernel v3 placement: items (cascade warps, sections + u = unit-gain form + T = TPDF finish + g = "
                    "source gain; d = dither warp, s = store warp) : IMAD.WIDE + other issue per frame:";
    char b[64];
    int macs[4] = {0, 0, 0, 0}, gen[4] = {0, 0, 0, 0}, other[4] = {0, 0, 0, 0};
    for (int k = 0; k < total; k++) {
        const Chain3Price p = chain3Price(plan, g, k);
        if (k < g.nCascade) {
            const ChainDesc& d = plan.chains[g.warpChain[k]];
            snprintf(b, sizeof b, " %d%s%s%s:%d+%d", g.warpNsec[k], g.warpUnit[k] ? "u" : "", g.warpFinal[k] && (d.satKind & 1) ? "T" : "",
                     g.warpSrc[k] < 0 && !(d.srcKind == SRC_LOAD_GAIN && d.srcArg == (1 << kMant)) ? "g" : "", p.macs, p.other);
        } else snprintf(b, sizeof b, " %s:%d+%d", k == g.nCascade ? "d" : "s", p.macs, p.other);
        s += b;
        macs[bin[k]] += p.macs; gen[bin[k]] += p.macsGeneral; other[bin[k]] += p.other;
    }
    s += "; sub-partition of each item ";
    for (int k = 0; k < total; k++) { snprintf(b, sizeof b, "%s%d", k ? "," : "", bin[k]); s += b; }
    snprintf(b, sizeof b, "; IMAD.WIDE per frame on sub-partitions 0-3: %d %d %d %d", macs[0], macs[1], macs[2], macs[3]);
    s += b;
    snprintf(b, sizeof b, ", every part general: %d %d %d %d", gen[0], gen[1], gen[2], gen[3]);
    s += b;
    snprintf(b, sizeof b, "; model cost (issue cycles per frame): %d %d %d %d\n", chain3BinCost(macs[0], other[0]), chain3BinCost(macs[1], other[1]),
             chain3BinCost(macs[2], other[2]), chain3BinCost(macs[3], other[3]));
    return s + b;
}

// Exact placement search.  Items with equal prices are one class; a bin is a count vector over the classes, and bins of
// equal size are filled in non-increasing order of their vectors, so every placement distinct up to interchangeable items and
// sub-partition relabelling is visited once (C2: 4229), pruned by the best placement so far.
struct Chain3Search {
    int nClass, nBin, slots[4];
    int macs[32], other[32], gen[32], otherGen[32], avail[32];   // per class: prices (planned, general form), items left
    int cur[4][32], best[4][32];                           // per bin: items of each class
    bool general;                                          // price every part in its general form
    int genBound;                                          // largest all-general bin cost a placement may have
    long long bestKey[2];                                  // largest bin cost, then the sum of squared bin costs

    int binCost(int q, bool gen_) const {
        int m = 0, o = 0;
        for (int c = 0; c < nClass; c++) { m += cur[q][c] * (gen_ ? gen[c] : macs[c]); o += cur[q][c] * (gen_ ? otherGen[c] : other[c]); }
        return chain3BinCost(m, o);
    }
    void fill(int q, int c, int room, long long maxCost, long long sumSq) {
        if (c == nClass) {
            if (room) return;
            if (q > 0 && slots[q] == slots[q - 1] &&
                std::lexicographical_compare(cur[q - 1], cur[q - 1] + nClass, cur[q], cur[q] + nClass)) return;
            if (binCost(q, true) > genBound) return;
            const long long cost = binCost(q, general);
            const long long k0 = std::max(maxCost, cost), k1 = sumSq + cost * cost;
            if (k0 > bestKey[0] || (q == nBin - 1 && k0 == bestKey[0] && k1 >= bestKey[1])) return;
            if (q == nBin - 1) {
                bestKey[0] = k0; bestKey[1] = k1;
                std::copy(&cur[0][0], &cur[0][0] + 4 * 32, &best[0][0]);
            } else fill(q + 1, 0, slots[q + 1], k0, k1);
            return;
        }
        for (int n = std::min(avail[c], room); n >= 0; n--) {
            cur[q][c] = n; avail[c] -= n;
            fill(q, c + 1, room - n, maxCost, sumSq);
            avail[c] += n; cur[q][c] = 0;
        }
    }
    long long run(bool general_, int genBound_) {
        general = general_; genBound = genBound_;
        bestKey[0] = bestKey[1] = LLONG_MAX;
        fill(0, 0, slots[0], 0, 0);
        return bestKey[0];
    }
};

// warps -> sub-partitions (hardware warp id % 4, tools/microbench_smsp.cu).  Item k is cascade warp k, then the dither warp,
// then the store warps; itemBin[k] = its sub-partition.  The placement minimises the largest sub-partition price in the
// planned forms, among the placements whose largest all-general price is the least any placement
// reaches: a CTA that a per-stream coefficient row sends back to the general form runs on the best all-general placement the
// prices know (C2: 55 55 65 65 IMAD.WIDE, no more than before the unit-gain form).
static void placeChain3Warps(const ChainPlan& plan, const Chain3Geom& g, int total, int* itemBin) {
    Chain3Search s{};
    s.nBin = std::min(total, 4);
    for (int q = 0; q < s.nBin; q++) s.slots[q] = (total - q + 3) / 4;
    int cls[32];
    for (int k = 0; k < total; k++) {
        const Chain3Price p = chain3Price(plan, g, k);
        int c = 0;
        while (c < s.nClass && !(s.macs[c] == p.macs && s.other[c] == p.other && s.gen[c] == p.macsGeneral && s.otherGen[c] == p.otherGeneral)) c++;
        if (c == s.nClass) { s.macs[c] = p.macs; s.other[c] = p.other; s.gen[c] = p.macsGeneral; s.otherGen[c] = p.otherGeneral; s.nClass++; }
        s.avail[c]++;
        cls[k] = c;
    }
    s.run(false, (int)s.run(true, INT_MAX));
    for (int k = 0; k < total; k++)
        for (int q = 0; q < s.nBin; q++)
            if (s.best[q][cls[k]] > 0) { s.best[q][cls[k]]--; itemBin[k] = q; break; }
}

bool planChain3Geometry(const ChainPlan& plan, int nStreams, int numSMs, Chain3Geom* geom) {
    if (!chain3Supports(plan)) return false;
    const int C = plan.h.nChains;
    int NS = envInt3("AVDSP_B200_NS3", 0);
    if (NS <= 0) NS = (nStreams + numSMs - 1) / numSMs;
    NS = std::max(1, std::min(NS, 32));
    int maxDelay = 0;
    for (int c = 0; c < C; c++) maxDelay = std::max(maxDelay, plan.chains[c].delayN);
    // Two shapes: cascades cut into parts of <= 4 sections (more, equal warps: the faster shape when it fits), else whole cascades
    for (int partMax : {envInt3("AVDSP_B200_PART3", 4), 8}) {
        if (partMax < 1 || partMax > 8) continue;
        if (plan.h.aluClass == ALU_F32 && partMax > 4) continue;      // the float form exists for parts of <= 4 sections
        struct Part { int chain, first, nsec, base, src, fin, unit; };
        Part parts[kChain3MaxWarps];
        int nParts = 0, gmax = 0, maxSec = 0;
        bool fits = true;
        Chain3Geom g{};
        for (int c = 0; c < C && fits; c++) {
            const int nsec = plan.chains[c].nsec, np = (nsec + partMax - 1) / partMax;
            // a SAT0DB_TPDF finish reads the dither ring (4 tiles) at the part's lag: at most two parts there; plain chains may be
            // cut further (C3: 16 sections = four parts of four), their lag only lengthens the row ring
            if (np > ((plan.chains[c].satKind & 1) ? 2 : 4)) { fits = false; break; }
            int first = 0, base = 0, prev = -1;
            for (int p = 0; p < np; p++) {
                if (nParts >= kChain3MaxWarps) { fits = false; break; }
                const int n = nsec / np + (p < nsec % np ? 1 : 0);          // near-equal parts, the longer ones first
                // the unit-gain form exists for the fixed-point parts of 3 and 4 sections (register checkpoint: partMax <= 4)
                bool unit = plan.h.aluClass == ALU_INT64 && partMax <= 4 && n >= 3;
                for (int k = first; k < first + n && unit; k++) {
                    const int32_t* cf = plan.pool + plan.chains[c].coefOff + 5 * k;
                    unit = cf[0] == (1 << kMantBQ) && (long long)cf[1] + cf[3] == -(1ll << kMantBQ) && (long long)cf[2] + cf[4] == 0;
                }
                parts[nParts] = {c, first, n, base, prev, p == np - 1, unit ? 1 : 0};
                prev = nParts++;
                first += n;
                maxSec = std::max(maxSec, n);
                gmax = std::max(gmax, base + n - 1);
                if (p == np - 1) g.chainLag[c] = base + n - 1;
                base += n - 1 + F3;                                       // the next part reads this part's row one tile later
            }
        }
        if (!fits) continue;
        const int maxThreads = maxSec > 4 ? kChain3MaxThreads : kChain3MaxThreadsParts;
        g.streamsPerCta = NS;
        g.floatFast = 1;          // float class: hardware convert + mul.rz.ftz on the source when every LOAD_GAIN gain is within [2^-30, 2^30]
        for (int c = 0; c < C; c++)
            if (plan.chains[c].srcKind == SRC_LOAD_GAIN) {
                const int ex = (int)(((uint32_t)plan.chains[c].srcArg >> 23) & 255u);
                if (ex != 0 && (ex < 127 - 30 || ex > 127 + 30)) g.floatFast = 0;
            }
        if (envInt3("AVDSP_B200_FLOAT_EXACT_HELPERS", 0)) g.floatFast = 0;
        g.nCascade = nParts;
        g.gmax = gmax;
        g.maxSec = maxSec;
        // (float class: the store warps also saturate and convert, measured best with four on C3-float: 5.27 ms against 5.40 with three)
        g.nStore = std::max(1, std::min(envInt3("AVDSP_B200_SW3", plan.h.aluClass == ALU_F32 ? 4 : 3), maxThreads / 32 - nParts - 1));
        g.threads = (nParts + 1 + g.nStore) * 32;
        if (g.threads > maxThreads) continue;
        // the cascades write steps of tile i+1 while the store warps still read window i back to (its first frame - longest delay)
        int R = 2 * F3;
        while (R < 2 * F3 + gmax + maxDelay) R <<= 1;
        g.postRing = R; g.postPitch = R + 1;
        g.rawPitchBytes = F3 * plan.h.nIn * 4 + 16;         // 16-byte aligned rows, 4-bank skew between streams
        g.rawStageBytes = NS * g.rawPitchBytes;
        // warps -> sub-partitions (hardware warp id % 4, tools/microbench_smsp.cu).  Every warp gets an issue cost per frame
        // (5 MACs + shift + saturation record per section; more for a SAT0DB_TPDF finish or a LOAD_GAIN; the dither and store
        // warps count too); longest-processing-time first, then pairwise swaps while they flatten the four sums.  C2 ends up
        // as (4T,4,3,helper) x 2 + (4,3,3,3) x 2: 8.66 ms per step against 9.08 with equal section counts per sub-partition
        // (both TPDF parts on one of them) -- the heaviest single warp sets the pace of its sub-partition.
        // Programs with unit-gain parts (C2) are placed by the exact search on measured prices instead (placeChain3Warps):
        // that search picks slower placements for C3 and C3-float (profiles/r7_chain3_ab.jsonl).
        // Cascade warp index w (rows, tables) is independent of the hardware warp id.
        for (int w = 0; w < nParts; w++) {
            g.warpChain[w] = parts[w].chain; g.warpFirstSec[w] = parts[w].first; g.warpNsec[w] = parts[w].nsec;
            g.warpBase[w] = parts[w].base; g.warpSrc[w] = parts[w].src; g.warpFinal[w] = parts[w].fin;
            g.warpUnit[w] = parts[w].unit;
            if (parts[w].fin) g.chainRow[parts[w].chain] = w;
        }
        {
            const int total = nParts + 1 + g.nStore;
            int slots[4];
            for (int q = 0; q < 4; q++) slots[q] = (total - q + 3) / 4;   // warp ids q, q+4, ... below total
            int itemCost[32], itemBin[32], order[32];
            for (int k = 0; k < total; k++) {
                order[k] = k;
                if (k >= nParts) { itemCost[k] = 8; continue; }              // helper warps: k == nParts dither, then store
                const ChainDesc& d = plan.chains[parts[k].chain];
                itemCost[k] = 5 * parts[k].nsec + 2;
                if (parts[k].fin && (d.satKind & 1)) itemCost[k] += 6;
                if (parts[k].src < 0 && !(d.srcKind == SRC_LOAD_GAIN && d.srcArg == (1 << kMant))) itemCost[k] += 2;
            }
            std::stable_sort(order, order + total, [&](int a, int b) { return itemCost[a] > itemCost[b]; });
            int binCost[4] = {0, 0, 0, 0}, used[4] = {0, 0, 0, 0};
            for (int k = 0; k < total; k++) {
                int best = -1;
                for (int q = 0; q < 4; q++) if (used[q] < slots[q] && (best < 0 || binCost[q] < binCost[best])) best = q;
                itemBin[order[k]] = best; used[best]++; binCost[best] += itemCost[order[k]];
            }
            for (int iter = 0; iter < 64; iter++) {
                int ba = -1, bb = -1; long long bestGain = 0;
                for (int a = 0; a < total; a++)
                    for (int b = a + 1; b < total; b++) {
                        const int qa = itemBin[a], qb = itemBin[b];
                        if (qa == qb || itemCost[a] == itemCost[b]) continue;
                        const int dlt = itemCost[a] - itemCost[b];             // a's bin loses dlt, b's bin gains it
                        const long long before = (long long)binCost[qa] * binCost[qa] + (long long)binCost[qb] * binCost[qb];
                        const long long after = (long long)(binCost[qa] - dlt) * (binCost[qa] - dlt) + (long long)(binCost[qb] + dlt) * (binCost[qb] + dlt);
                        if (before - after > bestGain) { bestGain = before - after; ba = a; bb = b; }
                    }
                if (ba < 0) break;
                const int qa = itemBin[ba], qb = itemBin[bb], dlt = itemCost[ba] - itemCost[bb];
                binCost[qa] -= dlt; binCost[qb] += dlt;
                itemBin[ba] = qb; itemBin[bb] = qa;
            }
            bool anyUnit = false;
            for (int k = 0; k < nParts; k++) anyUnit |= parts[k].unit != 0;
            if (anyUnit) placeChain3Warps(plan, g, total, itemBin);
            if (const char* ov = getenv("AVDSP_B200_BINS3")) {          // experiments: "b0,b1,..." = sub-partition of item k (parts, dither, stores)
                int k = 0;
                for (const char* q = ov; *q && k < total; q++) if (*q >= '0' && *q <= '3') itemBin[k++] = *q - '0';
                int cnt[4] = {0, 0, 0, 0};
                for (int kk = 0; kk < total; kk++) cnt[itemBin[kk]]++;
                for (int q = 0; q < 4; q++) if (cnt[q] != slots[q]) return false;
            }
            int next[4] = {0, 0, 0, 0};
            for (int k = 0; k < 32; k++) g.warpRole[k] = -1;
            // cascade index = part index k (rows follow the part order); hardware warp id = bin + 4 * position in the bin
            for (int k = 0; k < total; k++) {
                const int id = itemBin[k] + 4 * next[itemBin[k]]++;
                if (k < nParts) g.warpRole[id] = k; else g.warpRole[id] = -1 - (k - nParts);
            }
        }
        size_t bytes = 0;
        g.postOff = 0;
        for (int w = 0; w < nParts; w++) {                  // final parts: R-step ring (the delay line); hand-over rows: three tiles
            g.warpPitch[w] = g.warpFinal[w] ? g.postPitch : 3 * F3 + 1;
            g.warpRowOff[w] = (int)bytes; bytes += (size_t)NS * g.warpPitch[w] * 4;
        }
        g.tpdfOff = (int)bytes; bytes += (size_t)NS * TP3 * 4;
        g.ckOff = (int)bytes;   if (maxSec > 4) bytes += (size_t)(5 * maxSec + 2) * nParts * 32 * 4;   // short parts checkpoint in registers
        g.doneOff = (int)bytes; bytes += (size_t)kChain3MaxWarps * 4;
        bytes = (bytes + 15) & ~(size_t)15;
        g.mbarOff = (int)bytes; bytes += 16;
        bytes = (bytes + 127) & ~(size_t)127;
        g.rawOff = (int)bytes;  bytes += (size_t)2 * g.rawStageBytes;
        g.smemBytes = bytes + 16;
        if (g.smemBytes > 226 * 1024) continue;
        *geom = g;
        return true;
    }
    return false;
}

// bulk copies need interleaved, 16-byte friendly input rows; everything else is staged with plain copies
static bool chain3TmaOk(const ChainPlan& plan, const Chain2Args& a) {
    const int nIn = plan.h.nIn;
    return a.inChStride == 1 && a.inFrameStride == nIn && ((size_t)a.in & 15) == 0 && (a.inStreamStride & 3) == 0 && ((F3 * nIn * 4) & 15) == 0;
}

cudaError_t launchChain3(const ChainPlan& plan, const Chain3Geom& geom, const Chain2Args& args, cudaStream_t stream) {
    Chain3Geom g = geom;
    g.tma = chain3TmaOk(plan, args) ? 1 : 0;
    const int blocks = (args.nStreams + g.streamsPerCta - 1) / g.streamsPerCta;
    cudaError_t e;
    if (plan.h.aluClass == ALU_F32) {
        e = cudaFuncSetAttribute(k_chain3<4, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)g.smemBytes);
        if (e != cudaSuccess) return e;
        k_chain3<4, true><<<blocks, g.threads, g.smemBytes, stream>>>(plan, args, g);
    } else if (g.maxSec > 4) {
        e = cudaFuncSetAttribute(k_chain3<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)g.smemBytes);
        if (e != cudaSuccess) return e;
        k_chain3<8><<<blocks, g.threads, g.smemBytes, stream>>>(plan, args, g);
    } else {
        e = cudaFuncSetAttribute(k_chain3<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)g.smemBytes);
        if (e != cudaSuccess) return e;
        k_chain3<4><<<blocks, g.threads, g.smemBytes, stream>>>(plan, args, g);
    }
    return cudaGetLastError();
}

} // namespace avdsp

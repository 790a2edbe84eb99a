// kernels.h -- launch interfaces of the CUDA kernels (host side of kernel_*.cu).
#pragma once
#include <cuda_runtime.h>
#include <string>
#include <vector>
#include "plan.h"

namespace avdsp {

constexpr int kGenericThreads = 128;

// PCM addressing is fully strided (in words) so interleaved [stream][frame][ch] and planar
// [stream][ch][frame] layouts share the kernels.
struct GenericArgs {
    const int* in;  int* out;
    int* state;                 // [nStreams][stateWords]
    const int* bigPool;         // FIR taps / data tables in HBM
    int nStreams, nFrames;
    long long inStreamStride, outStreamStride;
    int inFrameStride, inChStride, outFrameStride, outChStride;
    int coreSel;                // -1: all cores; k: only core k (0-based)  -- dspRuntime_<fmt> compat path
    int period;                 // 0: canonical order; >0: ALSA plugin order with this period
    int stageState;             // filled by launchGeneric: the CTA works on a shared-memory copy of its streams' state blocks
    // second pass behind a fused kernel (api.cu): only the streams whose flag word is set run, from the state block the
    // snapshot holds (the state block itself behind the FIR kernels, which leave flagged streams untouched)
    const int* redo;            // [nStreams] or nullptr
    const int* snapshot;        // [nStreams][stateWords]
    // per-stream coefficient table (avdsp_b200_set_coefs) or nullptr: word [column][stream] at coefs[column * coefPitch + s]; a
    // BIQUADS micro-op's c is its first column, its sections step by coefStep (5 * the program's fs columns)
    const int* coefs;
    int coefPitch, coefStep;
    // per-stream FIR table (avdsp_b200_set_fir_taps) or nullptr: [stream][column], the stream at position s of the call reads
    // firTaps[s * firPitch + column]; firCol ([nOps], device): the column of FIR micro-op i's first tap (Lowered::firColOfOp)
    const int* firTaps;
    int firPitch;
    const int* firCol;
    unsigned coreInMask[kMaxCores], coreOutMask[kMaxCores];
};
cudaError_t launchGeneric(const GenericPlan& plan, const GenericArgs& args, cudaStream_t stream);

// ---- systolic chain kernel -------------------------------------------------------------------
// Lane table entry: which biquad section(s) a thread of the CTA owns.
struct ChainLane {
    int slot;        // streamLocal * nChains + chain, or -1 for an idle lane
    int depth;       // pipeline depth of this lane inside its chain (0 = head)
    int flags;       // bit0 head, bit1 tail
    int firstSec;    // index of the lane's first section inside the chain
};
// ---- warp-specialised systolic chain kernel (kernel_chain2.cu) -----------------------------------
struct Chain2Geom {
    int streamsPerCta;     // NS
    int secPerLane;        // K
    int tileFrames;        // F: steps between barriers (32 or 16)
    int gmax;              // largest frame offset of a cascade tail (longest cascade - 1)
    int secThreads;        // threads that own sections (multiple of 32, may be 0)
    int helpThreads;       // source / sink / dither threads (multiple of 32, >= 32)
    int helpersFirst;      // 1: helper warps get the low warp ids
    int floatFast;         // float class: LOAD_GAIN sources may use the hardware convert + mul.rz.ftz (gains checked on the host)
    int debugSkip;         // timing experiments only (AVDSP_B200_DEBUG_SKIP): bit0 skip sources, bit1 skip PRNG, bit2 skip sink
    int postRing;          // R: post ring length in steps (power of two >= F + gmax + longest delay)
    int xPitch, accPitch, postPitch, tpdfPitch;   // shared-memory row pitches (elements)
    int mbarOff, rawOff;   // byte offsets of the helper warps' mbarriers / the TMA-staged input tiles (0: none)
    // shared-memory map in BYTES (acc ring at 0) and per-stream block sizes, so that the helper warps form
    // every address with adds on constants instead of recomputing products of geometry values
    int xOff, postOff, tpdfOff, ridxOff, ckOff;
    int accStreamBytes, xStreamBytes, postStreamBytes, tpdfStreamBytes, rawStreamBytes;
    // byte offsets inside one stream's block, by STATIC index (constant-bank operands):
    int outRowOff[kFastTab];   // output channel j  -> its chain's post row
    int outPos4[kFastTab];     // output channel j  -> 4*(cascade lag - delay)
    int pPostOff[kFastTab];    // post-processed chain k -> its post row
    int pAccOff[kFastTab];     // post-processed chain k -> its acc row
    int srcXOff[kFastTab];     // source k -> its x row
    size_t smemBytes;
};
struct Chain2Args {
    const int* in;  int* out;
    int* state;
    const ChainLane* lanes;     // [secThreads]
    int nStreams, nFrames;
    long long inStreamStride, outStreamStride;
    int inFrameStride, inChStride, outFrameStride, outChStride;
    int* redo;                  // float class: [nStreams] flag words, set to 1 for a stream that has to be re-executed exactly (avdsp_dev.cuh, fltGuard)
    // exact second pass of the float class (k_chain2 only): the launch works on the streams listed in `map` (positions in the
    // call's stream range), as many as *countPtr says (device memory: the list is built by the pass before), with
    // dspMulFloatFloat as hardware product + integer fallback and the host's NaN rules on the adds
    const int* map;
    const int* countPtr;
    int exact;
    // per-stream coefficient table (avdsp_b200_set_coefs) or nullptr: [column][stream] words, coefs[column * coefPitch + p] for
    // the stream at position p of the call; the cascades load their coefficients from it instead of the plan
    const int* coefs;
    int coefPitch;
};
// before a float-class chain kernel, one launch: state blocks of the range -> snapshot, flags and list counter cleared
cudaError_t launchRedoPrepare(const int* state, int* snapshot, size_t words, int* flags, int nStreams, int* count, cudaStream_t stream);
// after a float-class chain kernel: list the flagged streams of the range and put their state blocks back to the snapshot
cudaError_t launchRedoCompact(const int* flags, int nStreams, int* list, int* count, int* state, const int* snapshot, int stateWords, cudaStream_t stream);
bool chainFloatCoefsInRange(const ChainPlan& plan);     // float class: every non-zero biquad coefficient within [2^-60, 2^7)
bool chain2Supports(const ChainPlan& plan);
bool planChain2Geometry(const ChainPlan& plan, int nStreams, int numSMs, Chain2Geom* geom, ChainLane* lanesOut /*[1024]*/);
cudaError_t launchChain2(const ChainPlan& plan, const Chain2Geom& geom, const Chain2Args& args, cudaStream_t stream);

// ---- DAG kernel (kernel_dag.cu): programs that route signals through the X/Y registers -------------------------------
constexpr int kDagMaxThreads = 384;         // up to 12 warps of 168 registers: whole cascades (<= 8 sections) per lane
struct DagGeom {
    int streamsPerCta;     // NS (<= 32): lane = stream, warp = node
    int threads, nStore;
    int tileFrames;        // frames per iteration (32, or 16 when that lets a CTA hold its share of the streams)
    int perStreamWords;    // one stream's block of rows in shared memory (odd)
    int rawOff, rawMask;   // staged input PCM, one row per channel: word offset inside a stream's block, frames - 1 (power of two)
    int tpdfOff, tpdfMask; // dither values
    int nRawOut;           // output channels that are DSP_LOAD_STORE copies (written by the staging warp)
    int rawOutCh[kIoSlots], rawOutSrc[kIoSlots];           // ... which ones, and the input channel each copies (-1: reads 0)
    int accMask[kMaxDagNodes];
    int staleOff;          // word offset (from the start of shared memory) of the stale-index notes for the store warps
    int tabOff;            // ... of the store warps' per-element table and the staging warp's frame table
    int accLoOff[kMaxDagNodes], accHiOff[kMaxDagNodes];       // 64-bit node values, two planes
    int postOff[kMaxDagNodes], postMask[kMaxDagNodes];        // finished s.31 outputs (the delay line behind the saturation)
    int aDlyOff[kMaxDagNodes], aDlyMask[kMaxDagNodes];        // private delay rows of the operands (DSP_DELAY on a sample, DSP_DELAY_DP)
    int bDlyOff[kMaxDagNodes], bDlyMask[kMaxDagNodes];
    size_t smemBytes;
};
struct Chain2Args;
bool planDagGeometry(const DagPlan& plan, int nStreams, int numSMs, DagGeom* geom);
cudaError_t launchDag(const DagPlan& plan, const DagGeom& geom, const Chain2Args& args, cudaStream_t stream);

// ---- register-resident cascade kernel (kernel_chain3.cu): lane = one whole cascade of one stream ------------------
constexpr int kChain3MaxChains = 10;        // chains of a program the kernel takes
constexpr int kChain3MaxWarps = 16;         // cascade warps of a CTA (chains, or parts of chains)
constexpr int kChain3MaxThreads = 384;      // whole cascades (<= 8 sections): 3 warps per sub-partition (16384 registers each) = 168 registers per thread
constexpr int kChain3MaxThreadsParts = 512; // parts of <= 4 sections: 4 warps per sub-partition = 128 registers per thread
struct Chain3Geom {
    int streamsPerCta;     // NS (<= 32): lane = stream inside a cascade warp
    int nCascade;          // cascade warps
    int nStore;            // store warps
    int gmax;              // largest lag of a warp's tail (sections are skewed in time, parts run a tile behind each other)
    int maxSec;            // longest part (selects the kernel instance)
    int threads;           // (nCascade + 1 + nStore) * 32
    int postRing;          // R: row ring length in steps (power of two >= 2 tiles + gmax + longest delay)
    int postPitch;         // R + 1
    int rawPitchBytes, rawStageBytes;     // staged input tiles: bytes per stream row / per stage (2 stages)
    int postOff, tpdfOff, ckOff, doneOff, mbarOff, rawOff;   // shared-memory map (bytes)
    int tma;               // filled per launch: the caller's input buffer allows bulk copies (else plain staged copies)
    int floatFast;         // float class: the source may use the hardware convert + mul.rz.ftz (gains checked on the host)
    // cascade warp -> what it runs (placed on the sub-partitions through warpRole, kernel_chain3.cu placeChain3Warps)
    int warpChain[kChain3MaxWarps], warpFirstSec[kChain3MaxWarps], warpNsec[kChain3MaxWarps];
    int warpBase[kChain3MaxWarps];        // step offset of the part: its section k works on frame t - base - k at step t
    int warpSrc[kChain3MaxWarps];         // -1: the PCM tile; else the warp whose row feeds this part
    int warpFinal[kChain3MaxWarps];       // last part of its chain
    // the program's coefficients put every section of the part in the unit-gain form (kernel_chain3.cu unitStep: 2 MACs per section
    // instead of 5).  Placement and the trace use it; the warp itself decides from the words it loads (a per-stream table may differ)
    int warpUnit[kChain3MaxWarps];
    int warpRowOff[kChain3MaxWarps];      // byte offset of the warp's rows [stream][pitch] in shared memory
    int warpPitch[kChain3MaxWarps];       // words per row: R + 1 (final parts: the post ring) or 3 tiles + 1 (hand-over rows)
    int warpRole[32];                     // hardware warp id -> cascade warp index (>= 0), -1 dither warp, -2-k store warp k
    int chainRow[kChain3MaxChains];       // chain -> row (= warp) of its final part
    int chainLag[kChain3MaxChains];       // chain -> lag of its final part's tail
    size_t smemBytes;
};
bool chain3Supports(const ChainPlan& plan);
bool planChain3Geometry(const ChainPlan& plan, int nStreams, int numSMs, Chain3Geom* geom);
std::string chain3PlacementTrace(const ChainPlan& plan, const Chain3Geom& geom);   // the trace line of the warp placement
cudaError_t launchChain3(const ChainPlan& plan, const Chain3Geom& geom, const Chain2Args& args, cudaStream_t stream);

// ---- time-parallel mixer / delay / dither kernel (kernel_mix.cu) -----------------------------------
// Everything the three kernels need, flattened by OUTPUT channel (static indices -> constant-bank operands).
struct MixPlan {
    int nIn, nOut, nChains, nInPad;
    int stateWords, auxOff;
    int hasCalc, tpdfDither, tpdfDataOff, tpdfShift, anyTpdf;
    int storeMask, maxDelay;
    int cDelay[kFastTab], cDelayOff[kFastTab], cMuxOff[kFastTab], cOut[kFastTab];      // per chain
    int oChain[kFastTab], oDelay[kFastTab], oDelayOff[kFastTab], oFlags[kFastTab], oGain[kFastTab], oSatGain[kFastTab],
        oKind[kFastTab], oSrcCh[kFastTab], oMatRow[kFastTab], oDelayBytes[kFastTab], oDelayPcmBytes[kFastTab];   // per output channel
    int uniform, uFlags;                                                                // all outputs: dense row + the same flags
    int mat[kFastTab * kFastTab];                                                        // dense gain rows [chain][input]
};
struct MixArgs {
    const int* in;  int* out;
    int* state;
    int* tpdfBuf;               // [nStreams][nFrames] dither values of this launch (scratch)
    int nStreams, nFrames;
    long long inStreamStride, outStreamStride;
    int inFrameStride, inChStride, outFrameStride, outChStride;
    int vecIn, vecOut;          // 16-byte paths usable (interleaved + aligned)
    int tileFrames, winFrames;  // filled by launchMix
};
bool buildMixPlan(const ChainPlan& plan, MixPlan* out, std::string* why);
void mixJumpMatrix(long long steps, unsigned* out /*[128*4]*/);
constexpr int kMixJumpLevels = 8;                 // up to 256 jump-ahead segments per stream: level b holds M^(2L * 2^b)
void mixPrngSegments(const MixPlan& M, const MixArgs& A, int numSMs, int* J, int* L);
cudaError_t launchMix(const MixPlan& M, MixArgs A, const unsigned* dJump, int J, int L, int numSMs, cudaStream_t stream, int* launches);

// ---- time-parallel FIR kernels (kernel_fir.cu) ---------------------------------------------------
struct FirArgs {
    const int* in;  int* out;
    int* state;
    const int* bigPool;         // taps (Q4.28 ints or float bits)
    int nStreams, nFrames;
    long long inStreamStride, outStreamStride;
    int inFrameStride, inChStride, outFrameStride, outChStride;
    // per-stream FIR table (avdsp_b200_set_fir_taps) or nullptr: the stream at position p of the call convolves with
    // taps[p * tapPitch + FirPath::tapCol ...]; skip (or nullptr): [nStreams] flag words, set for a stream the FIR kernels leave
    // alone (float rows with a tap below 2^-60: the interpreter runs it, see launchRun)
    const int* taps;
    int tapPitch;
    const int* skip;
};
// exact kernels: int64 accumulation (any order is exact) / float in the reference's tap order
cudaError_t launchFir(const FirPlan& plan, const FirArgs& args, int numSMs, cudaStream_t stream, int* launches);
cudaError_t launchFirState(const FirPlan& plan, const FirArgs& args, cudaStream_t stream);      // delay-line update only

// ---- Toeplitz-GEMM FIR on tcgen05 tensor cores (kernel_fir_tc.cu) -------------------------------------
enum FirTcKind : int { FIRTC_I8 = 0 /* DSP_FORMAT 2: 8-bit limbs, bit-exact */, FIRTC_TF32 = 1 /* DSP_FORMAT 3: 3xTF32, stated tolerance */ };
int firTcHistory(const FirPlan& plan);
void firTcBuildTaps(const FirPlan& plan, int kind, const int32_t* bigPool, std::vector<unsigned char>* out);
size_t firTcWorkspaceBytes(const FirPlan& plan, int kind, int nStreams, int nFrames);
cudaError_t launchFirTc(const FirPlan& plan, int kind, const FirArgs& args, const unsigned char* dTaps, unsigned char* workspace,
                        cudaStream_t stream, int* launches);
// per-stream form (FIRTC_I8, a per-stream FIR table): Toeplitz planes of every stream built on the device from the table
// ([stream][column], nCols columns), then pack + GEMM (128 outputs x 64 output blocks of one stream per CTA) + delay lines
size_t firTcPerTapsBytes(const FirPlan& plan, int nStreams);
size_t firTcPerWorkspaceBytes(const FirPlan& plan, int nStreams, int nFrames);
cudaError_t launchFirTcBuildTaps(const FirPlan& plan, const int* table, int nCols, int nStreams, unsigned char* out, cudaStream_t stream);
cudaError_t launchFirTcPer(const FirPlan& plan, const FirArgs& args, const unsigned char* dTaps, unsigned char* workspace,
                           cudaStream_t stream, int* launches);

} // namespace avdsp

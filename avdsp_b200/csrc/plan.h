// plan.h -- the lowered form of one AVDSP program: what the host decoder (decoder.cpp) produces
// and what the CUDA kernels consume.  Plans are passed to kernels BY VALUE as __grid_constant__
// parameters, i.e. they live in the constant bank for the duration of a launch: every micro-op
// fetch, gain, coefficient and delay length is a warp-uniform constant-cache read, and no
// process-global __constant__ symbol is needed (several programs can be live at once, unlike the
// reference whose tables are file-scope globals, runtime/dsp_runtime.c:36-38,103-110).
//
// Per-stream mutable state lives in HBM as one block of `stateWords` int32 per stream ("AoS"):
//   [0, dataSize)            the reference's data area, SAME word offsets (dsp_runtime.c:137-141)
//   [auxOff, auxOff+8)       what the reference keeps in globals: xoshiro s[4], tpdfValue,
//                            tpdfRandom, current global dither, pad            (dsp_tpdf.h:11-33)
//   [memOff, memOff+2*nMem)  the 64-bit PARAM words targeted by LOAD_MEM/STORE_MEM, which the
//                            reference mutates inside the code area (dsp_runtime.c:750-766)
#pragma once
#include <cstdint>
#include "wire.h"

namespace avdsp {

// ---------------------------------------------------------------- error codes (C-ABI) ---------
// The first six are the reference's own (dsp_runtime.c:116-195).
enum Err : int {
    ERR_NO_HEADER   = -1,   // also: unknown sampling frequency (dspRuntimeReset)
    ERR_FS_RANGE    = -2,
    ERR_NO_CORE     = -3,
    ERR_CHECKSUM    = -4,
    ERR_OPCODE_NEW  = -5,
    ERR_TOO_LARGE   = -6,
    ERR_FORMAT      = -7,   // ours: unsupported DSP_FORMAT or program encoded for another format
    ERR_UNSUPPORTED = -8,   // ours: opcode / program shape the executor rejects (e.g. DSP_SINE)
    ERR_ARG         = -9,
    ERR_CUDA        = -10,
    ERR_MALFORMED   = -11,  // ours: pointer/offset walks outside the program or data area
    ERR_PLAN_SIZE   = -12,  // ours: lowered plan exceeds the kernel-parameter budget
    ERR_ENCODER_OLD = -13,  // ours: file made by an encoder older than 0x102 (11-word header, other opcode layouts)
};

enum AluClass : int { ALU_INT64 = 0, ALU_F32 = 1, ALU_F64 = 2 };

constexpr int kMaxCores   = 16;
constexpr int kMaxOps     = 320;
constexpr int kMaxPool    = 2304;
constexpr int kAuxWords   = 8;
enum { AUX_S0 = 0, AUX_S1, AUX_S2, AUX_S3, AUX_TPDF_VALUE, AUX_TPDF_RANDOM, AUX_DITHER, AUX_PAD };

// One lowered opcode.  `op` keeps the reference opcode number; operands are fully resolved:
// relative code pointers became immediates / pool offsets, the fs column is picked, delay times are
// samples, bypassed biquads and zero-length delays are dropped.
struct MicroOp {
    uint16_t op;
    uint16_t n;        // count (mux pairs, biquad sections, load_store pairs)
    int32_t  a, b, c;
};

struct PlanHeader {
    int32_t format;            // DSP_FORMAT 2..6
    int32_t aluClass;          // AluClass
    int32_t sampleInt;         // 1: io[] holds int32 s.31, 0: float (formats 5/6)
    int32_t nCores;
    int32_t coreStart[kMaxCores + 1];   // ops[coreStart[c] .. coreStart[c+1])
    int32_t nIn, nOut;
    uint8_t inIdx[kIoSlots];   // io slot of input channel k   (ascending slot order)
    uint8_t outIdx[kIoSlots];  // io slot of output channel k
    int32_t defaultDither;
    int32_t dataSize;          // words of the reference data area
    int32_t stateWords;        // per-stream block size (multiple of 4)
    int32_t auxOff, memOff, nMem;
    int32_t nOps, nPool;
};

struct GenericPlan {
    PlanHeader h;
    MicroOp    ops[kMaxOps];
    int32_t    pool[kMaxPool];
};

// ---------------------------------------------------------------- chain plan ------------------
// A "chain" is one independent signal path   source -> [biquad cascade] -> [gain] -> saturate
// (+dither,+gain) -> [delay] -> store(s).   Programs made only of such chains (C2, C3, C5 and most
// crossovers) run on the systolic chain kernel instead of the generic interpreter.
constexpr int kMaxChains     = 48;
constexpr int kMaxChainPool  = 2560;
constexpr int kMaxChainStores = 4;
constexpr int kFastTab       = 16;     // entries of the flattened helper tables (chain2 handles programs within them)
enum { PF_SECTIONS = 1, PF_GAIN = 2, PF_SAT_TPDF = 4, PF_SAT_GAIN = 8, PF_RAW = 16 /* DSP_LOAD_STORE pass-through */,
       PF_DELAY_FIRST = 32 /* cascade -> DELAY -> SAT0DB*: the ring holds the low word of the accumulator, the finish runs on the delayed value */ };
constexpr int kMaxMemCopy = 8;

enum ChainSrc : int { SRC_LOAD = 0, SRC_LOAD_GAIN = 1, SRC_LOAD_MUX = 2,
                      SRC_RAW = 3 /* a DSP_LOAD_STORE pair: the output is the input sample, untouched (no saturation, no STORE mask) */ };
enum ChainSat : int { SAT_PLAIN = 0, SAT_TPDF = 1, SAT_GAIN = 2, SAT_TPDF_GAIN = 3 };

struct ChainDesc {
    uint8_t  srcKind, satKind, hasGain, nStores;
    uint8_t  storeCh[kMaxChainStores];   // OUTPUT CHANNEL numbers (not io slots)
    int32_t  srcId;           // chains with sections: index of the (deduplicated) source feeding the head, else -1
    int32_t  accRow;          // chains whose sink needs the full 64-bit accumulator: row in the acc ring, else -1.
                              // accRow < 0 && nsec > 0: "direct" chain (cascade -> SAT0DB): the tail's y1 IS the s.31 output
    int16_t  nsec;            // total biquad sections (concatenated consecutive BIQUADS ops)
    int16_t  srcCh;           // SRC_LOAD/LOAD_GAIN: INPUT CHANNEL number;  LOAD_MUX: pair count
    int32_t  srcArg;          // LOAD_GAIN: gain bits;  LOAD_MUX: pool offset of (inputChannel, gain) pairs
    int32_t  muxStateOff;     // LOAD_MUX: data offset of the stored 64-bit result, else -1
    int32_t  coefOff;         // pool offset of 5*nsec coefficients (b0 b1 b2 a1-1 a2 per section)
    int32_t  secStateOff;     // pool offset of nsec data-area offsets (6 words each, dsp_biquadSTD.h:45)
    int32_t  coefColOff;      // pool offset of nsec coefficient-table columns (Lowered::coefWords: the section's b0 at this fs)
    int32_t  gainBits;        // optional GAIN between cascade and saturation
    int32_t  satGainBits;     // SAT0DB_GAIN / SAT0DB_TPDF_GAIN
    int32_t  delayOff, delayN;// ring in the data area ([index][n samples]); delayN==0: none
    int32_t  delayFirst;      // 1: the DELAY sits between the cascade and the saturation (osx/dacdiy1.bin)
};

struct ChainHeader {
    int32_t format, aluClass, sampleInt;
    int32_t nChains, nIn, nOut;
    int32_t hasTpdfCalc, tpdfDither, tpdfDataOff;   // DSP_TPDF_CALC at the start of core 1
    int32_t storeDither;                            // dither whose mask applies to every STORE
    int32_t tpdfShift;                              // 28 - dither + 1 (dsp_tpdf.h:63)
    int32_t dataSize, stateWords, auxOff;
    int32_t maxSec;                                 // longest cascade
    int32_t totalSec;                               // sum of nsec
    int32_t nPool;
    int32_t nSrc;                                   // distinct sources among chains that have sections
    int32_t srcChain[kMaxChains];                   // a chain that carries source k's description
    int32_t nUnwritten;                             // output channels no path stores to (they read 0)
    int32_t nDelayFirst;                            // paths with the DELAY in front of the saturation (k_chain2 only)
    int32_t nRaw;                                   // DSP_LOAD_STORE pass-through paths
    // cascades handed from one core to the next through a MEM word (source -> BIQUADS -> STORE_MEM m ... LOAD_MEM m -> BIQUADS ->
    // ...) are inlined into their consumers; after a launch MEM m must hold what the producer stored last: the accumulator of
    // its last section, which the section lanes leave in the data area anyway
    int32_t nMemCopy, memCopyDst[kMaxMemCopy], memCopySrc[kMaxMemCopy];
    int32_t nAcc;                                   // acc-ring rows per stream
    int32_t nProc;                                  // chains the sink has to post-process (everything but direct chains)
    int32_t procChain[kMaxChains];
    int32_t chainOfOut[kIoSlots];                   // output channel -> chain (or -1: channel never written => 0)
    int32_t outOff[kIoSlots];                       // output channel -> (cascade lag - delay): frame f is read from post-ring step f+outOff
    // flattened copies of the descriptors the helper warps touch every tile, indexed by small STATIC indices so
    // that they become constant-bank operands (no loads, no registers): post-processed chains and sources 0..7
    int32_t pChain[kFastTab], pLag[kFastTab], pAccRow[kFastTab], pFlags[kFastTab], pGain[kFastTab], pSatGain[kFastTab], pDelayN[kFastTab];
    int32_t sKind[kFastTab], sCh[kFastTab], sArg[kFastTab];
};

struct ChainPlan {
    ChainHeader h;
    ChainDesc   chains[kMaxChains];
    int32_t     pool[kMaxChainPool];
};

// ---------------------------------------------------------------- DAG plan (kernel_dag.cu) ----
// Programs that route signals through the X/Y register pair -- subtractive crossovers (`COPYXY ... SWAPXY ... SUBYX`:
// dspprogs/crossoverLV6.c, oktodac_fabriceo.c), forks (`COPYXY ... SWAPXY`: crossover2x2lfe.c), sums of MEM words
// (`LOAD_MEM; LOAD_MEM; ADDXY`) -- are not sets of independent chains: a path may start from a combination of what other
// paths computed in the same frame.  The decoder executes X/Y symbolically and turns such a program into a small DAG:
// every NODE is  input expression -> [biquad cascade] -> [finish: gain / saturate / dither -> post-saturation delay -> stores],
// the expression being  V = A [+|- B]  [>> shift] [* gain]  over OPERANDS (an input sample, optionally delayed (DSP_DELAY)
// and scaled; the 64-bit value of an earlier node, optionally delayed (DSP_DELAY_DP); a LOAD_MUX sum).
constexpr int kMaxDagNodes  = 10;
constexpr int kMaxDagStores = 6;
constexpr int kMaxDagPool   = 1536;
enum DagOpdKind : int { OPD_NONE = 0 /* the value 0 */, OPD_RAW = 1, OPD_NODE = 2, OPD_MUX = 3 };
enum DagFinish  : int { FIN_NONE = 0 /* no output of its own */, FIN_SAT = 1 /* [GAIN] -> SAT0DB[_TPDF][_GAIN] */,
                        FIN_TRUNC = 2 /* DSP_STORE of an unsaturated value: its low word (dsp_runtime.c:610-633) */ };
struct DagOperand {
    int32_t kind;                // DagOpdKind
    int32_t arg;                 // RAW: input CHANNEL (-1: slot nobody feeds, reads 0); NODE: node index; MUX: pool offset of (channel, gain) pairs
    int32_t n;                   // MUX: pair count
    int32_t hasGain, gain;       // RAW: X = sample * gain (LOAD_GAIN, or LOAD [DELAY] GAIN);  NODE: unused
    int32_t delayKind;           // 0 none; 1 DSP_DELAY on the raw sample, before the gain (ring of int32); 2 DSP_DELAY_DP on a node value (ring of int64)
    int32_t delayN, delayOff;    // samples; data-area offset of the ring ([index | line], dsp_runtime.c:769-824)
    int32_t muxStateOff;         // MUX: data offset of the stored 64-bit sum, else -1
};
struct DagNode {
    DagOperand a, b;
    int32_t comb;                // 0: V = A;  +1: V = A + B;  -1: V = A - B
    int32_t postShift;           // > 0: V >>= postShift (DSP_SHIFT with a negative count) after the combination
    int32_t hasPostGain, postGain;   // then V *= gain (DSP_GAIN, 64 x 32 wrapping)
    int32_t nsec, coefOff, secStateOff, coefColOff;   // cascade: x = V >> 28 (dsp_runtime.c:831); pool offsets as in ChainDesc
    int32_t exportAcc;           // a later node (or a MEM word) takes this node's 64-bit value
    int32_t memOff;              // DSP_STORE_MEM target (state offset) or -1
    int32_t finKind;             // DagFinish
    int32_t finHasGain, finGain; // DSP_GAIN between the cascade and the saturation
    int32_t satKind, satGain;    // ChainSat
    int32_t delayN, delayOff;    // DSP_DELAY behind the saturation (ring of s.31 values), 0: none
    int32_t depth;               // tiles behind the input: 1 + deepest NODE operand
    int32_t nStores;
    int32_t storeCh[kMaxDagStores], storeDelayed[kMaxDagStores];   // OUTPUT CHANNEL; 1: the STORE sits behind the DELAY
};
struct DagPlan {
    int32_t nNodes, nIn, nOut, nPool;
    int32_t dataSize, stateWords, auxOff;
    int32_t hasTpdfCalc, tpdfDither, tpdfDataOff, storeDither, tpdfShift;
    int32_t maxDepth, maxSec;
    // output channel -> where its samples come from: node >= 0 (its post row, `delayed`: read behind the node's DELAY),
    // -1: nobody stores it (reads 0), -2: DSP_LOAD_STORE copy of input channel outRaw[ch] (no saturation, no STORE mask)
    int32_t outNode[kIoSlots], outDelayed[kIoSlots], outRaw[kIoSlots];
    DagNode nodes[kMaxDagNodes];
    int32_t pool[kMaxDagPool];
};

// ---------------------------------------------------------------- FIR plan -------------------
// DSP_FIR taps live in HBM ("big pool"); one entry per FIR micro-op.
struct FirDesc {
    int32_t tapsOff;     // word offset into the big pool
    int32_t length;      // taps
    int32_t stateOff;    // data-area offset of the delay line (length words)
};

// Programs made only of paths   LOAD|LOAD_GAIN -> FIR (convolution) -> [GAIN] -> SAT0DB[_GAIN] -> STORE(s)
// (room-correction / linear-phase crossover programs: BASELINE config C4) run on the time-parallel FIR
// kernels (kernel_fir.cu) instead of the per-frame interpreter.
constexpr int kMaxFirPaths = 16;
constexpr int kMaxFirTaps  = 8192;
struct FirPath {
    int32_t srcKind, srcCh, srcArg;      // ChainSrc; INPUT CHANNEL number (-1: reads 0); LOAD_GAIN gain bits
    int32_t tapsOff, length, stateOff;   // FirDesc
    int32_t flags, gainBits, satGainBits;// PF_GAIN / PF_SAT_GAIN
    int32_t nStores, storeCh[kMaxChainStores];   // OUTPUT CHANNEL numbers
    int32_t tapCol;                      // per-stream FIR table column of the first tap at this fs (Lowered::firTapWords)
};
struct FirPlan {
    int32_t aluClass, nPaths, nIn, nOut;
    int32_t stateWords, storeMask;
    int32_t maxLen;                      // longest impulse
    int32_t nUnwritten;                  // output channels no path stores to (they read 0)
    int32_t unwritten[kIoSlots];
    FirPath paths[kMaxFirPaths];
};

} // namespace avdsp

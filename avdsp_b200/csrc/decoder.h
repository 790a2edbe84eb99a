// decoder.h -- host-side front half of the executor: validate an AVDSP program exactly like
// dspRuntimeInit/dspRuntimeReset (runtime/dsp_runtime.c:116-195) and lower its opcode stream
// (runtime/dsp_runtime.c:302-1314 is the semantics being lowered) into plans (plan.h).
#pragma once
#include <cstdint>
#include <memory>
#include <string>
#include <vector>
#include "plan.h"

namespace avdsp {

struct CoreInfo {
    int coreWord;      // index of the DSP_CORE word (or 0 when the program has none)
    int beginWord;     // first executable opcode (dspFindCoreBegin)
    uint32_t usedIn, usedOut;
};

struct Lowered {
    // identity
    int format = 0, fs = 0, fsIndex = 0, fsRel = 0, nFreq = 0;
    int totalLength = 0, dataSize = 0, defaultDither = 0;
    std::vector<int32_t> words;          // private copy of the program (totalLength words)
    std::vector<CoreInfo> cores;
    // plans
    GenericPlan gen{};
    bool chainOk = false;
    std::string chainWhyNot;
    ChainPlan chain{};
    bool dagOk = false;                  // X/Y dataflow program that maps to a DAG of cascades (kernel_dag.cu)
    std::string dagWhyNot;
    std::shared_ptr<DagPlan> dag;      // re-lowering allocates a new one (copies of a Lowered may share the old)
    std::vector<int32_t> bigPool;        // FIR taps / data tables (device: HBM)
    std::vector<FirDesc> firs;
    bool firOk = false;                  // program maps to the time-parallel FIR kernels (kernel_fir.cu)
    std::string firWhyNot;
    FirPlan fir{};
    // true when no data flows from one core to another (MEM words, io slots, the TPDF value / dither table): then the ALSA
    // plugin's core-major loop nest (linux/avdsp_plugin.c:95-142) and the canonical frame-major order give identical results
    // for every period size, and a plugin-order request can run on the fused kernels
    bool orderIndependent = false;
    std::string orderWhy;
    // MEM words (LOAD_MEM / STORE_MEM targets inside the code area)
    std::vector<int> memWord;            // code word index of each slot
    // biquad coefficient words: b0 b1 b2 a1 a2 of every section of every DSP_BIQUADS parameter block, for every fs column,
    // bypassed blocks included, ascending.  The columns of the per-stream coefficient table (avdsp_b200_set_coefs); a lowered
    // BIQUADS micro-op's `c` is the column of its first section's b0 at the current fs, section k at c + 5 * nFreq * k.
    std::vector<int32_t> coefWords;
    bool coefTableOk = true;             // every lowered section follows that column pattern (blocks that overlap do not)
    // FIR tap words: t + 1 .. t + lw of every DSP_FIR entry that is a convolution (length word lw > 0, lw >> 16 == 0), for every
    // fs column, ascending, each word once.  The columns of the per-stream FIR table (avdsp_b200_set_fir_taps); a lowered FIR
    // convolution's column (firColOfOp[its micro-op index], FirPath::tapCol) is that of its first tap at the current fs, tap k at
    // that + k.  Kept beside the plan, not in it: the plan-only kernels never see it.
    std::vector<int32_t> firTapWords;
    std::vector<int32_t> firColOfOp;     // [nOps]: column of a FIR convolution micro-op, -1 for every other micro-op
    // human readable trace of the lowering (replaces the reference's DSP_PRINTF=2 opcode trace)
    std::string trace;
};

// returns totalLength (>0) or a negative Err.  `maxWords` is the caller's buffer size in words as
// passed to dspRuntimeInit (size check -6); pass a huge value to skip.
int decodeProgram(const int32_t* prog, int progWords, int maxWords, int format, int fs,
                  int defaultDither, Lowered* out, std::string* err);

// Re-read only the parameter words of an already decoded program (host edited gains / delays /
// biquad coefficients in place; dump-file workflow, encoder/dsp_encoder.c:476-503).
int relowerProgram(const int32_t* prog, int progWords, Lowered* inout, std::string* err);

// reference helpers kept at the boundary (runtime/dsp_runtime.c:42-77)
int findCoreWord(const int32_t* prog, int numCore /*1-based*/);   // -1 when absent
int findCoreBeginWord(const int32_t* prog, int coreWord);

} // namespace avdsp

// instance.h -- the executor instance behind the opaque avdsp_b200_t of include/avdsp_b200.h (private to csrc/).
#pragma once
#include <cuda_runtime.h>
#include <map>
#include <memory>
#include <string>
#include <vector>
#include "../../include/avdsp_b200.h"
#include "decoder.h"
#include "kernels.h"

// A per-stream table of program words (avdsp_b200_set_coefs, avdsp_b200_set_fir_taps): one row per stream, column c holds
// word (L.*words)[c]; d == nullptr: none.  Variants (set_param on other words) keep their own plans and read the same table.
struct StreamTable {
    decltype(&avdsp::Lowered::coefWords) words;     // the column list: &Lowered::coefWords or &Lowered::firTapWords
    bool streamMajor;           // [stream][column] (rows arrive in this layout: one copy), else [column][stream]
    const char* noun;           // what a column holds, for messages
    int* d = nullptr;
    int* dStage = nullptr; size_t stageWords = 0;   // [column][stream]: HOST rows on their way to the table
    // word (stream s, column c) lives at d[s * streamStride + c * colStride]
    size_t streamStride(size_t nCols) const { return streamMajor ? nCols : 1; }
    size_t colStride(size_t nStreams) const { return streamMajor ? 1 : nStreams; }
};

// What one program word list needs on one device: its lowering, the kernels that can take it and their plan data there.  Owns
// its buffers (no copies), freed on the device uploadPlanData put them on; one that never uploaded makes no CUDA call (describe).
struct Plans {
    avdsp::Lowered L;
    int* dBig = nullptr; size_t bigWords = 0;
    int* dFirCol = nullptr;         // L.firColOfOp on the device: the FIR-table column of each micro-op (k_generic with a FIR table)
    avdsp::ChainLane* dLanes2 = nullptr;
    avdsp::Chain2Geom geom2{};
    bool chain2Usable = false;      // kernel_chain2.cu (v2: warp-specialised, the default)
    avdsp::Chain3Geom geom3{};
    bool chain3Usable = false;      // kernel_chain3.cu (v3: one cascade per lane; the common crossover / EQ shape at batch width)
    avdsp::DagGeom geomDag{};
    bool dagUsable = false;         // kernel_dag.cu (X/Y dataflow programs: a DAG of cascades, node per warp)
    avdsp::MixPlan mix{};
    bool mixUsable = false;         // kernel_mix.cu (time-parallel: programs without biquads)
    bool firUsable = false;         // kernel_fir.cu (time-parallel FIR paths)
    unsigned char* dFirTaps = nullptr;              // kernel_fir_tc.cu: pre-swizzled Toeplitz taps blobs
    std::string trace;
    int planDevice = -1;            // where the buffers above live (-1: nothing uploaded)
    Plans() = default;
    Plans(const Plans&) = delete; Plans& operator=(const Plans&) = delete;
    ~Plans() {
        if (planDevice < 0) return;
        cudaSetDevice(planDevice);
        cudaFree(dBig); cudaFree(dFirCol); cudaFree(dLanes2); cudaFree(dFirTaps);       // cudaFree(nullptr) does nothing
    }
};

// An instance is its program's plans plus the streams that run them.
struct avdsp_b200 : Plans {
    int device = 0, numSMs = 148;
    int nStreams = 0;
    std::vector<int32_t> seeds;
    int* dState = nullptr;
    int* dMemInit = nullptr;
    int* dSeeds = nullptr;
    int lastChainVariant = 0;       // 2 / 3: which chain kernel the last AVDSP_B200_KERNEL_CHAIN launch used
    unsigned char* dFirWs = nullptr; size_t firWsBytes = 0;     // kernel_fir_tc.cu: the packed-sample workspace
    unsigned* dJump = nullptr; int jumpL = -1;      // PRNG jump matrix for segments of jumpL draws
    int* dTpdf = nullptr; size_t tpdfWords = 0;     // scratch dither values of a launch
    // float class of the chain kernels: per-stream "re-execute me exactly" flags and the state snapshot the interpreter's second
    // pass starts from (avdsp_dev.cuh fltGuard; launchRun).  Indexed by the instance's stream number: disjoint runs do not collide.
    int* dRedo = nullptr; int* dSnap = nullptr; int* dRedoList = nullptr; int* dRedoCount = nullptr;   // + the compacted list of a run (by instance stream number)
    int period = 0, kernelSel = AVDSP_B200_KERNEL_AUTO, lastKernel = 0;
    long long launches = 0;
    cudaStream_t stream = nullptr;          // for the synchronous calls
    // Calls on one instance are STREAM-ORDERED by the library: launches share per-instance scratch (dither rows, FIR workspace,
    // PRNG jump matrices) and continue each other's state, so every launch waits for the previous one's event whatever CUDA
    // stream the caller passed, and every host-side mutation (reload_params, reset, get/set_state) synchronises on it first.
    cudaEvent_t evLast = nullptr;
    // host-memspace staging: a few slots of device buffers + copy streams
    static constexpr int kSlots = 3;
    cudaStream_t slotStream[kSlots] = {nullptr, nullptr, nullptr};
    int* slotIn[kSlots] = {nullptr, nullptr, nullptr};
    int* slotOut[kSlots] = {nullptr, nullptr, nullptr};
    size_t slotInWords = 0, slotOutWords = 0;
    cudaEvent_t evIn[kSlots] = {nullptr, nullptr, nullptr}, evKernel[kSlots] = {nullptr, nullptr, nullptr}, evOut[kSlots] = {nullptr, nullptr, nullptr};
    void* pcmRaw = nullptr; int* pcmIn = nullptr; int* pcmOut = nullptr; size_t pcmRawBytes = 0, pcmInWords = 0, pcmOutWords = 0;
    // multi-device instance (avdsp_b200_create_multi): this object only carries the decoded program; the streams live in
    // one single-device instance per GPU, contiguous balanced ranges (stream s of the whole = stream s - shardFirst[k] of shard k)
    std::vector<avdsp_b200*> shards;
    std::vector<int> shardFirst;       // [nShards + 1]
    // per-stream parameter overrides (avdsp_b200_set_param): variantOf[s] == 0: the program as loaded, v > 0: the plans of the
    // patched words in variants[v - 1].  Empty variantOf: no override anywhere.  Streams keep their state blocks whatever variant
    // they run.  A variant is released only once the instance is quiesced (quiesce, freeAll): launches read its plan data.
    std::vector<int> variantOf;
    std::vector<std::unique_ptr<Plans>> variants;
    // runs of streams on different variants are independent launches: they go out on a few forked streams and join the caller's
    static constexpr int kVarStreams = 32;
    cudaStream_t varStream[kVarStreams] = {};
    cudaEvent_t varEv[kVarStreams] = {};
    cudaEvent_t evFork = nullptr;
    // per-stream coefficient table: [column][stream], so that the chain, DAG and generic kernels' lane = stream loads coalesce
    StreamTable coefTab{&avdsp::Lowered::coefWords, false, "biquad coefficient"};
    // per-stream FIR table: [stream][column], so that a k_fir CTA stages its stream's taps as one coalesced run.  Float programs
    // (ALU_F32) also keep one flag word per stream: set when the stream's row holds a non-zero tap below 2^-60, which the FIR
    // kernels cannot multiply exactly (launchRun).
    StreamTable firTab{&avdsp::Lowered::firTapWords, true, "FIR tap"};
    int* dFirFlags = nullptr;
    // DSP_FORMAT 2 with a FIR table: every stream's Toeplitz limb planes for the per-stream tensor-core form (kernel_fir_tc.cu),
    // built on the device before the first such launch after the rows changed (valid = false)
    unsigned char* dFirTcPer = nullptr; bool firTcPerValid = false;
    bool firTcPerFailed = false;       // their allocation failed once: this instance runs k_fir with its table
    int numaNode = -1;                 // host NUMA node next to `device` (-1: unknown)
    std::map<void*, size_t> hostAllocs;   // avdsp_b200_host_alloc: pointer -> bytes
};


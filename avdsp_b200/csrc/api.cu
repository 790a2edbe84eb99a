// api.cu -- the C ABI of the executor (include/avdsp_b200.h): instance management, state in HBM,
// kernel selection, host<->device staging, and the reference's own entry points as a per-frame
// compatibility path.  No CPU fallback exists: without a CUDA device every compute call fails.
//
// Reference behaviour mirrored here (citations: /root/reference/module_avdsp/):
//   dspRuntimeInit / dspRuntimeReset   runtime/dsp_runtime.c:150-195 / :116-145
//   dspFindCore / dspFindCoreBegin     runtime/dsp_runtime.c:42-77
//   dspTpdfInit (PRNG seeding)         runtime/dsp_tpdf.h:85-99
//   dsp_transfer (the batched caller)  linux/avdsp_plugin.c:71-163
#include "../../include/avdsp_b200.h"
#include "decoder.h"
#include "kernels.h"
#include "host_numa.h"
#include <cuda_runtime.h>
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

using namespace avdsp;

static thread_local std::string g_lastError;
static int setErr(int code, const std::string& msg) { g_lastError = msg; return code; }
static int cudaErr(cudaError_t e, const char* what) {
    return setErr(AVDSP_B200_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
}
#define NO_MULTI(h, what) do { if (!(h)->shards.empty()) return setErr(AVDSP_B200_ERR_UNSUPPORTED, what " takes a single-device instance (device buffers belong to one GPU)"); } while (0)
#define CU(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return cudaErr(e_, #call); } while (0)

// ---------------------------------------------------------------------------------------------
// state initialisation == dspRuntimeReset for every stream
__global__ void k_init_state(int* __restrict__ state, int W, int auxOff, int memOff, int nMem,
                             const int* __restrict__ memInit, const int* __restrict__ seeds,
                             int defaultDither, int nStreams) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= nStreams) return;
    int* st = state + (size_t)s * W;
    const unsigned u = seeds ? (unsigned)seeds[s] : 0u;
    int* aux = st + auxOff;
    // dspTpdfInit, runtime/dsp_tpdf.h:93-97
    aux[AUX_S0] = (int)(u | 1u);
    aux[AUX_S1] = (int)__funnelshift_l(u | 8u, u | 8u, 7);
    aux[AUX_S2] = (int)__funnelshift_l(u | 16u, u | 16u, 11);
    aux[AUX_S3] = (int)__funnelshift_l(u | 24u, u | 24u, 17);
    aux[AUX_TPDF_VALUE] = 0;
    aux[AUX_TPDF_RANDOM] = (int)u;
    aux[AUX_DITHER] = defaultDither;
    aux[AUX_PAD] = 0;
    for (int k = 0; k < 2 * nMem; k++) st[memOff + k] = memInit[k];
}

// integer-pipe microbenchmark: 8 independent chains of DATA-DEPENDENT accumulating IMAD.WIDE per thread (the
// multiplicand is the running accumulator's low word, so nothing can be hoisted or strength-reduced).  Same
// kernel as tools/microbench_int.cu mode 0; SASS: one IMAD.WIDE R, R, R, R per MAC.
__device__ __forceinline__ int peakLo32(long long v) { int l, h2; asm("mov.b64 {%0,%1}, %2;" : "=r"(l), "=r"(h2) : "l"(v)); (void)h2; return l; }
__global__ void __launch_bounds__(256) k_int_peak(long long* out, int iters, int a0, int b0) {
    long long acc[8];
    const int b = b0 + (int)blockIdx.x;
#pragma unroll
    for (int k = 0; k < 8; k++) acc[k] = (long long)(a0 + k + (int)threadIdx.x) * 0x100000001ll;
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int k = 0; k < 8; k++) acc[k] = acc[k] + (long long)peakLo32(acc[k]) * (long long)b;
    }
    long long s = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) s ^= acc[k];
    if (s == 0x123456789abcdefll) out[0] = s;     // practically never true; keeps the chains alive
}

// float-pipe microbenchmark for the FP32 roofline of the float kernels: 8 independent chains per thread of the
// reference's non-fused MAC, acc = add.rn(acc, mul.rz.ftz(x, c)) -- scalar (FMUL + FADD) or packed (FMUL2 + FADD2,
// two MACs per instruction pair).  Counts MACs.
template <int PACKED>
__global__ void __launch_bounds__(256) k_f32_peak(float* out, int iters, float c0) {
    // the multiplicand is the running accumulator, so neither instruction can be hoisted: acc += rz(acc * c), c < 0
    const float c = c0 - 1e-7f * (float)blockIdx.x;
    if constexpr (PACKED == 0) {
        float acc[8];
#pragma unroll
        for (int k = 0; k < 8; k++) acc[k] = 1e3f * (float)(k + 1 + (int)threadIdx.x);
        for (int i = 0; i < iters; i++) {
#pragma unroll
            for (int k = 0; k < 8; k++) {
                float p; asm volatile("mul.rz.ftz.f32 %0, %1, %2;" : "=f"(p) : "f"(acc[k]), "f"(c));
                asm volatile("add.rn.f32 %0, %0, %1;" : "+f"(acc[k]) : "f"(p));
            }
        }
        float s = 0.f;
#pragma unroll
        for (int k = 0; k < 8; k++) s += acc[k];
        if (s == 123.456f) out[0] = s;
    } else {
        unsigned long long acc[8], cc;
        asm("mov.b64 %0, {%1, %1};" : "=l"(cc) : "f"(c));
#pragma unroll
        for (int k = 0; k < 8; k++) {
            const float a = 1e3f * (float)(k + 1 + (int)threadIdx.x);
            asm("mov.b64 %0, {%1, %1};" : "=l"(acc[k]) : "f"(a));
        }
        for (int i = 0; i < iters; i++) {
#pragma unroll
            for (int k = 0; k < 8; k++) {
                unsigned long long p;
                asm volatile("mul.rz.ftz.f32x2 %0, %1, %2;" : "=l"(p) : "l"(acc[k]), "l"(cc));
                asm volatile("add.rn.f32x2 %0, %0, %1;" : "+l"(acc[k]) : "l"(p));
            }
        }
        unsigned long long s = 0;
#pragma unroll
        for (int k = 0; k < 8; k++) s ^= acc[k];
        if (s == 0x123456789abcdefull) out[0] = 1.f;
    }
}

// ALSA sample formats -> s.31 (linux/avdsp_plugin.c:109-121)
__global__ void k_widen_pcm(const unsigned char* __restrict__ src, int fmt, int* __restrict__ dst, size_t n) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int v;
    if (fmt == AVDSP_B200_PCM_S16) v = (int)((const short*)src)[i] << 16;
    else { const unsigned char* p = src + 3 * i; v = (int)(((unsigned)p[0] << 8) | ((unsigned)p[1] << 16) | ((unsigned)p[2] << 24)); }
    dst[i] = v;
}

// Rows of the coefficient table, [n][nCoef] (row s = stream first + s, avdsp_b200_set_coefs), into the table, [nCoef][pitch]:
// a transpose through 32 x 32 tiles so that both the row reads and the column writes coalesce.  block (32, 8), grid (stream
// tiles, column tiles).
__global__ void __launch_bounds__(256) k_coef_scatter(int* __restrict__ tab, int pitch, int first, int n, int nCoef, const int* __restrict__ rows) {
    __shared__ int t[32][33];
    const int s0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
    for (int j = threadIdx.y; j < 32; j += 8) {
        const int s = s0 + j, c = c0 + threadIdx.x;
        if (s < n && c < nCoef) t[j][threadIdx.x] = rows[(size_t)s * nCoef + c];
    }
    __syncthreads();
    for (int j = threadIdx.y; j < 32; j += 8) {
        const int c = c0 + j, s = s0 + threadIdx.x;
        if (s < n && c < nCoef) tab[(size_t)c * pitch + first + s] = t[threadIdx.x][j];
    }
}

// Exactness flags of the per-stream FIR table (float programs): flags[first + s] = 1 when row s holds a non-zero tap below
// 2^-60, the bound under which the FIR kernels' products can come near 2^-126 and differ from dspMulFloatFloat (the rule
// buildFirPlan applies to the program's own taps).  Every fs column counts.  One warp per stream.
__global__ void __launch_bounds__(256) k_fir_tap_flags(const int* __restrict__ tab, int nCols, int first, int n, int* __restrict__ flags) {
    const int s = (int)(blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32), lane = (int)(threadIdx.x & 31);
    if (s >= n) return;
    const int* row = tab + (size_t)(first + s) * nCols;
    bool tiny = false;
    for (int c = lane; c < nCols; c += 32) {
        const unsigned ex = ((unsigned)row[c] >> 23) & 255u;
        tiny |= ex != 0u && ex < 127u - 60u;
    }
    tiny = __any_sync(0xFFFFFFFFu, tiny);
    if (lane == 0) flags[first + s] = tiny ? 1 : 0;
}

#include "instance.h"

static int quiesce(avdsp_b200* h);
static int resetShards(avdsp_b200* h, int fs, const int32_t* seeds, int defaultDither);

// Host-only half of plan preparation: which kernels can take the program, their CTA geometries, the lowering trace.
static void planGeometries(Plans& p, int nStreams, int numSMs, std::vector<ChainLane>* lanes2) {
    const Lowered& L = p.L;
    p.chain2Usable = false;
    lanes2->assign(1024, ChainLane{});
    if (L.chainOk && chain2Supports(L.chain)) p.chain2Usable = planChain2Geometry(L.chain, nStreams, numSMs, &p.geom2, lanes2->data());
    p.chain3Usable = p.chain2Usable && planChain3Geometry(L.chain, nStreams, numSMs, &p.geom3);
    p.mixUsable = false;
    if (L.chainOk) { std::string why; p.mixUsable = buildMixPlan(L.chain, &p.mix, &why); }
    p.firUsable = L.firOk;
    p.dagUsable = L.dagOk && L.dag && planDagGeometry(*L.dag, nStreams, numSMs, &p.geomDag);
    char line[512];
    p.trace = L.trace;
    if (p.firUsable) {
        snprintf(line, sizeof line, "time-parallel FIR kernel: usable (%d paths, longest impulse %d taps)\n", L.fir.nPaths, L.fir.maxLen);
        p.trace += line;
    } else if (!L.firs.empty()) p.trace += "FIR kernel not used: " + L.firWhyNot + "\n";
    if (p.mixUsable) p.trace += "time-parallel mix kernel: usable (no biquad in any path)\n";
    if (p.chain2Usable) {
        snprintf(line, sizeof line, "chain kernel v2 geometry: %d streams/CTA, %d sections/lane, tile %d frames, gmax %d, %d section threads + %d helper threads, %d sources, %zu B smem\n",
                 p.geom2.streamsPerCta, p.geom2.secPerLane, p.geom2.tileFrames, p.geom2.gmax, p.geom2.secThreads, p.geom2.helpThreads, L.chain.h.nSrc, p.geom2.smemBytes);
        p.trace += line;
    }
    if (p.chain3Usable) {
        snprintf(line, sizeof line, "chain kernel v3 geometry: %d streams/CTA (lane = one cascade part of one stream), %d cascade warps of <= %d sections + 1 dither warp + %d store warps, largest lag %d frames, row ring %d steps, %zu B smem; parts (chain:first+n@base):",
                 p.geom3.streamsPerCta, p.geom3.nCascade, p.geom3.maxSec, p.geom3.nStore, p.geom3.gmax, p.geom3.postRing, p.geom3.smemBytes);
        p.trace += line;
        int macs = 0, algMacs = 0, unitSecs = 0;
        for (int w = 0; w < p.geom3.nCascade; w++) {
            snprintf(line, sizeof line, " %d:%d+%d@%d%s", p.geom3.warpChain[w], p.geom3.warpFirstSec[w], p.geom3.warpNsec[w], p.geom3.warpBase[w],
                     p.geom3.warpUnit[w] ? "u" : "");
            p.trace += line;
            algMacs += 5 * p.geom3.warpNsec[w];
            macs += (p.geom3.warpUnit[w] ? 2 : 5) * p.geom3.warpNsec[w];
            if (p.geom3.warpUnit[w]) unitSecs += p.geom3.warpNsec[w];
        }
        snprintf(line, sizeof line, "; unit-gain form (u) on %d sections: %d IMAD.WIDE per frame executed, %d algorithmic", unitSecs, macs, algMacs);
        p.trace += line;
        p.trace += "; sub-partitions (sections of the cascade warps on hardware warps q, q+4, ..; d = dither warp, s = store warp):";
        for (int q = 0; q < 4; q++) {
            p.trace += q ? " |" : " ";
            for (int id = q; id < p.geom3.threads / 32; id += 4) {
                const int role = p.geom3.warpRole[id];
                if (role >= 0) snprintf(line, sizeof line, " %d", p.geom3.warpNsec[role]);
                else snprintf(line, sizeof line, " %s", role == -1 ? "d" : "s");
                p.trace += line;
            }
        }
        p.trace += "\n";
        p.trace += chain3PlacementTrace(L.chain, p.geom3);
    }
    if (p.dagUsable) {
        snprintf(line, sizeof line, "DAG kernel geometry: %d nodes (depth %d, longest cascade %d sections), %d streams/CTA, %d threads, tiles of %d frames, input rows of %d frames, %d words/stream, %zu B smem%s\n",
                 L.dag->nNodes, L.dag->maxDepth, L.dag->maxSec, p.geomDag.streamsPerCta, p.geomDag.threads, p.geomDag.tileFrames, p.geomDag.rawMask + 1, p.geomDag.perStreamWords,
                 p.geomDag.smemBytes, (p.chain2Usable || p.mixUsable || p.firUsable) ? " (another fused kernel takes this program first)" : "");
        p.trace += line;
    } else if (!L.dagOk && !p.chain2Usable && !p.mixUsable && !p.firUsable) p.trace += "DAG kernel not used: " + L.dagWhyNot + "\n";
    if (!p.chain2Usable && !p.mixUsable) {
        const bool coefRange = L.chainOk && L.chain.h.aluClass == ALU_F32 && !chainFloatCoefsInRange(L.chain);
        snprintf(line, sizeof line, "chain kernels not used: %s\n",
                 coefRange ? "a biquad coefficient lies outside [2^-60, 2^7): the float class could not bound its products (exactness guard), the interpreter runs this program"
                           : L.chainOk ? "geometry does not fit" : L.chainWhyNot.c_str());
        p.trace += line;
    }
}

static int uploadPlanData(Plans& p, int device, int nStreams, int numSMs) {
    cudaSetDevice(device);
    p.planDevice = device;
    const Lowered& L = p.L;
    // big pool (FIR taps, data tables)
    if (p.dBig) { cudaFree(p.dBig); p.dBig = nullptr; }
    p.bigWords = L.bigPool.size();
    if (p.bigWords) {
        CU(cudaMalloc(&p.dBig, p.bigWords * 4));
        CU(cudaMemcpy(p.dBig, L.bigPool.data(), p.bigWords * 4, cudaMemcpyHostToDevice));
    }
    if (p.dFirCol) { cudaFree(p.dFirCol); p.dFirCol = nullptr; }
    if (!L.firColOfOp.empty()) {
        CU(cudaMalloc(&p.dFirCol, L.firColOfOp.size() * 4));
        CU(cudaMemcpy(p.dFirCol, L.firColOfOp.data(), L.firColOfOp.size() * 4, cudaMemcpyHostToDevice));
    }
    std::vector<ChainLane> lanes2;
    planGeometries(p, nStreams, numSMs, &lanes2);
    if (p.chain2Usable) {
        if (!p.dLanes2) CU(cudaMalloc(&p.dLanes2, 1024 * sizeof(ChainLane)));
        CU(cudaMemcpy(p.dLanes2, lanes2.data(), 1024 * sizeof(ChainLane), cudaMemcpyHostToDevice));
    }
    if (p.dFirTaps) { cudaFree(p.dFirTaps); p.dFirTaps = nullptr; }
    if (p.firUsable) {
        std::vector<unsigned char> blobs;
        firTcBuildTaps(L.fir, L.fir.aluClass == ALU_INT64 ? FIRTC_I8 : FIRTC_TF32, L.bigPool.data(), &blobs);
        CU(cudaMalloc(&p.dFirTaps, blobs.size()));
        CU(cudaMemcpy(p.dFirTaps, blobs.data(), blobs.size(), cudaMemcpyHostToDevice));
    }
    return 0;
}

// p's own words lowered at another rate / default dither into *nl (the multi-device parent takes only this half)
static int decodeAt(const Plans& p, int fs, int defaultDither, Lowered* nl) {
    std::string err;
    const int rc = decodeProgram(p.L.words.data(), (int)p.L.words.size(), 0x7FFFFFFF, p.L.format, fs, defaultDither, nl, &err);
    return rc < 0 ? setErr(rc, err) : rc;
}

// p re-planned at another rate / default dither for instance h's device and batch; its state layout may not change
static int replanAt(Plans& p, int fs, int defaultDither, const avdsp_b200* h) {
    Lowered nl;
    const int rc = decodeAt(p, fs, defaultDither, &nl); if (rc < 0) return rc;
    if (nl.gen.h.stateWords != p.L.gen.h.stateWords) return setErr(AVDSP_B200_ERR_ARG, "state layout changed on reset");
    p.L = std::move(nl);
    return uploadPlanData(p, h->device, h->nStreams, h->numSMs);
}

static int initState(avdsp_b200* h) {
    cudaSetDevice(h->device);
    const PlanHeader& P = h->L.gen.h;
    const size_t words = (size_t)h->nStreams * P.stateWords;
    CU(cudaMemsetAsync(h->dState, 0, words * 4, h->stream));
    std::vector<int32_t> memInit(2 * std::max(P.nMem, 1), 0);
    for (int k = 0; k < P.nMem; k++) {   // initial MEM values come from the program bytes (SURVEY.md A.5-7)
        memInit[2 * k] = h->L.words[h->L.memWord[k]];
        memInit[2 * k + 1] = h->L.words[h->L.memWord[k] + 1];
    }
    if (h->dMemInit) { cudaFree(h->dMemInit); h->dMemInit = nullptr; }
    CU(cudaMalloc(&h->dMemInit, memInit.size() * 4));
    CU(cudaMemcpyAsync(h->dMemInit, memInit.data(), memInit.size() * 4, cudaMemcpyHostToDevice, h->stream));
    if (!h->seeds.empty()) {
        if (!h->dSeeds) CU(cudaMalloc(&h->dSeeds, (size_t)h->nStreams * 4));
        CU(cudaMemcpyAsync(h->dSeeds, h->seeds.data(), (size_t)h->nStreams * 4, cudaMemcpyHostToDevice, h->stream));
    }
    const int th = 128;
    k_init_state<<<(h->nStreams + th - 1) / th, th, 0, h->stream>>>(h->dState, P.stateWords, P.auxOff, P.memOff, P.nMem, h->dMemInit,
                                                                     h->seeds.empty() ? nullptr : h->dSeeds, P.defaultDither, h->nStreams);
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(h->stream));
    return 0;
}

static void freeTable(StreamTable& t) {
    if (t.d) cudaFree(t.d);
    if (t.dStage) cudaFree(t.dStage);
    t.d = t.dStage = nullptr; t.stageWords = 0;
}

static void freeAll(avdsp_b200* h) {
    if (!h) return;
    for (auto& kv : h->hostAllocs) { cudaHostUnregister(kv.first); hostFreePlaced(kv.first, kv.second); }
    h->hostAllocs.clear();
    if (!h->shards.empty()) {
        for (avdsp_b200* sh : h->shards) freeAll(sh);
        delete h;
        return;
    }
    if (h->evLast) cudaEventSynchronize(h->evLast);
    cudaSetDevice(h->device);
    if (h->dState) cudaFree(h->dState);
    if (h->dMemInit) cudaFree(h->dMemInit);
    if (h->dSeeds) cudaFree(h->dSeeds);
    if (h->dJump) cudaFree(h->dJump);
    if (h->dTpdf) cudaFree(h->dTpdf);
    if (h->dRedo) cudaFree(h->dRedo);
    if (h->dSnap) cudaFree(h->dSnap);
    if (h->dRedoList) cudaFree(h->dRedoList);
    if (h->dRedoCount) cudaFree(h->dRedoCount);
    if (h->dFirWs) cudaFree(h->dFirWs);
    freeTable(h->coefTab);
    freeTable(h->firTab);
    if (h->dFirFlags) cudaFree(h->dFirFlags);
    if (h->dFirTcPer) cudaFree(h->dFirTcPer);
    if (h->pcmRaw) cudaFree(h->pcmRaw);
    if (h->pcmIn) cudaFree(h->pcmIn);
    if (h->pcmOut) cudaFree(h->pcmOut);
    for (int k = 0; k < avdsp_b200::kSlots; k++) {
        if (h->slotIn[k]) cudaFree(h->slotIn[k]);
        if (h->slotOut[k]) cudaFree(h->slotOut[k]);
        if (h->slotStream[k]) cudaStreamDestroy(h->slotStream[k]);
        if (h->evIn[k]) cudaEventDestroy(h->evIn[k]);
        if (h->evKernel[k]) cudaEventDestroy(h->evKernel[k]);
        if (h->evOut[k]) cudaEventDestroy(h->evOut[k]);
    }
    if (h->evLast) { cudaEventSynchronize(h->evLast); cudaEventDestroy(h->evLast); }
    for (int k = 0; k < avdsp_b200::kVarStreams; k++) {
        if (h->varStream[k]) { cudaStreamSynchronize(h->varStream[k]); cudaStreamDestroy(h->varStream[k]); }
        if (h->varEv[k]) cudaEventDestroy(h->varEv[k]);
    }
    if (h->evFork) cudaEventDestroy(h->evFork);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
}

extern "C" {

const char* avdsp_b200_last_error(void) { return g_lastError.c_str(); }

int avdsp_b200_create(avdsp_b200_t** out, const int32_t* prog, int progWords, int fs, int format,
                      int nStreams, const int32_t* seeds, int defaultDither, int device) {
    if (!out) return setErr(AVDSP_B200_ERR_ARG, "out is NULL");
    *out = nullptr;
    if (nStreams < 1) return setErr(AVDSP_B200_ERR_ARG, "nStreams must be >= 1");
    std::unique_ptr<avdsp_b200, void (*)(avdsp_b200*)> h(new avdsp_b200, freeAll);
    std::string err;
    const int rc = decodeProgram(prog, progWords, 0x7FFFFFFF, format, fs, defaultDither, &h->L, &err);
    if (rc < 0) return setErr(rc, err);
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return setErr(AVDSP_B200_ERR_CUDA, std::string("no CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0") +
                                               " (avdsp_b200 has no CPU fallback)");
    if (device < 0 || device >= ndev) return setErr(AVDSP_B200_ERR_ARG, "device ordinal out of range");
    h->device = device;
    h->nStreams = nStreams;
    CU(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    h->numSMs = prop.multiProcessorCount;
    { char bus[64] = {0}; if (cudaDeviceGetPCIBusId(bus, sizeof bus, device) == cudaSuccess) h->numaNode = numaNodeOfPci(bus); }
    if (seeds) h->seeds.assign(seeds, seeds + nStreams);
    CU(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
    CU(cudaEventCreateWithFlags(&h->evLast, cudaEventDisableTiming));
    const size_t words = (size_t)nStreams * h->L.gen.h.stateWords;
    CU(cudaMalloc(&h->dState, std::max<size_t>(words, 1) * 4));
    int r = uploadPlanData(*h, device, nStreams, h->numSMs); if (r < 0) return r;
    r = initState(h.get()); if (r < 0) return r;
    g_lastError.clear();
    *out = h.release();
    return rc;
}

void avdsp_b200_destroy(avdsp_b200_t* h) { freeAll(h); }

int avdsp_b200_describe(const int32_t* prog, int progWords, int fs, int format, int defaultDither, int nStreams, int numSMs,
                        char* out, int outLen) {
    if (!out || outLen < 1 || nStreams < 1 || numSMs < 1) return setErr(AVDSP_B200_ERR_ARG, "bad argument");
    Plans p;                                                 // host-only: decode + lower + plan, nothing touches CUDA
    std::string err;
    const int rc = decodeProgram(prog, progWords, 0x7FFFFFFF, format, fs, defaultDither, &p.L, &err);
    if (rc < 0) return setErr(rc, err);
    std::vector<ChainLane> lanes2;
    planGeometries(p, nStreams, numSMs, &lanes2);
    snprintf(out, (size_t)outLen, "%s", p.trace.c_str());
    return rc;
}

int avdsp_b200_reset(avdsp_b200_t* h, int fs, const int32_t* seeds, int defaultDither) {
    if (!h) return setErr(AVDSP_B200_ERR_ARG, "NULL instance");
    if (!h->shards.empty()) return resetShards(h, fs, seeds, defaultDither);
    { const int q = quiesce(h); if (q < 0) return q; }
    if (fs != h->L.fs || defaultDither != h->L.defaultDither) {
        const int r = replanAt(*h, fs, defaultDither, h); if (r < 0) return r;
        // the per-stream Toeplitz planes follow this rate's tap blocks (and their size its longest impulse)
        if (h->dFirTcPer) { cudaFree(h->dFirTcPer); h->dFirTcPer = nullptr; }
        h->firTcPerValid = h->firTcPerFailed = false;
        for (auto& v : h->variants)                           // the overrides stay; their plans follow the new rate / dither
            { const int vr = replanAt(*v, fs, defaultDither, h); if (vr < 0) return vr; }
    }
    if (seeds) h->seeds.assign(seeds, seeds + h->nStreams); else h->seeds.clear();
    return initState(h);
}

int avdsp_b200_io_map(const avdsp_b200_t* h, int* nIn, int* inIdx, int* nOut, int* outIdx) {
    if (!h) return setErr(AVDSP_B200_ERR_ARG, "NULL instance");
    const PlanHeader& P = h->L.gen.h;
    if (nIn) *nIn = P.nIn;
    if (nOut) *nOut = P.nOut;
    if (inIdx) for (int k = 0; k < P.nIn; k++) inIdx[k] = P.inIdx[k];
    if (outIdx) for (int k = 0; k < P.nOut; k++) outIdx[k] = P.outIdx[k];
    return 0;
}

int avdsp_b200_set_order(avdsp_b200_t* h, int period) {
    if (!h || period < 0) return setErr(AVDSP_B200_ERR_ARG, "bad period");
    for (avdsp_b200* sh : h->shards) sh->period = period;
    h->period = period; return 0;
}
int avdsp_b200_set_kernel(avdsp_b200_t* h, int which) {
    if (!h || which < 0 || which > AVDSP_B200_KERNEL_DAG) return setErr(AVDSP_B200_ERR_ARG, "bad kernel selector");
    for (avdsp_b200* sh : h->shards) sh->kernelSel = which;
    h->kernelSel = which; return 0;
}
int avdsp_b200_last_kernel(const avdsp_b200_t* h) { return !h ? 0 : h->shards.empty() ? h->lastKernel : h->shards[0]->lastKernel; }
int avdsp_b200_last_chain_variant(const avdsp_b200_t* h) {
    if (h && !h->shards.empty()) h = h->shards[0];
    return (h && h->lastKernel == AVDSP_B200_KERNEL_CHAIN) ? h->lastChainVariant : 0;
}
long long avdsp_b200_launch_count(const avdsp_b200_t* h) {
    if (!h) return 0;
    long long n = h->launches;
    for (const avdsp_b200* sh : h->shards) n += sh->launches;
    return n;
}
int avdsp_b200_state_words(const avdsp_b200_t* h) { return h ? h->L.gen.h.stateWords : 0; }
int avdsp_b200_data_size(const avdsp_b200_t* h) { return h ? h->L.gen.h.dataSize : 0; }
int avdsp_b200_aux_offset(const avdsp_b200_t* h) { return h ? h->L.gen.h.auxOff : 0; }
int avdsp_b200_mem_offset(const avdsp_b200_t* h) { return h ? h->L.gen.h.memOff : 0; }
int avdsp_b200_num_mem(const avdsp_b200_t* h) { return h ? h->L.gen.h.nMem : 0; }
int avdsp_b200_mem_word(const avdsp_b200_t* h, int k) { return (h && k >= 0 && k < (int)h->L.memWord.size()) ? h->L.memWord[k] : -1; }
int avdsp_b200_num_streams(const avdsp_b200_t* h) { return h ? h->nStreams : 0; }
int avdsp_b200_num_cores(const avdsp_b200_t* h) { return h ? h->L.gen.h.nCores : 0; }
const char* avdsp_b200_trace(const avdsp_b200_t* h) { return h ? h->trace.c_str() : ""; }

} // extern "C"

// One launch over streams [first, first+n) with device buffers.  coreSel/plan override serve the
// dspRuntime_<fmt> compatibility path.
// `pl`: the plans the streams run (the instance's own, or a variant a per-stream parameter override created, see
// avdsp_b200_set_param); state, scratch, tables and bookkeeping are the instance's.
// ordered = false: the caller (launchRange, runs of variants on forked streams) has done the instance's stream ordering itself.
static int launchRun(avdsp_b200* h, const Plans& pl, const int* in, int* out, int nFrames, int layout, int first, int n,
                     cudaStream_t stream, int coreSel, const GenericPlan* planOverride, int cap, bool ordered = true) {
    if (nFrames == 0 || n == 0) return 0;
    const GenericPlan& G = planOverride ? *planOverride : pl.L.gen;
    const PlanHeader& P = G.h;
    const int nIn = P.nIn, nOut = P.nOut;
    if (cap <= 0) cap = nFrames;            // frames the buffers are laid out for (>= nFrames: staging slots are reused for a shorter last chunk)
    long long inSS, outSS; int inFS, inCS, outFS, outCS;
    if (layout == AVDSP_B200_INTERLEAVED) {
        inSS = (long long)cap * nIn; inFS = nIn; inCS = 1;
        outSS = (long long)cap * nOut; outFS = nOut; outCS = 1;
    } else if (layout == AVDSP_B200_PLANAR) {
        inSS = (long long)cap * nIn; inFS = 1; inCS = cap;
        outSS = (long long)cap * nOut; outFS = 1; outCS = cap;
    } else return setErr(AVDSP_B200_ERR_ARG, "unknown layout");
    int* st = h->dState + (size_t)first * P.stateWords;
    const int* coefs = h->coefTab.d ? h->coefTab.d + first : nullptr;     // per-stream coefficient table, positioned like the state blocks
    const int nTapCols = (int)h->L.firTapWords.size();
    const int* firTaps = h->firTab.d ? h->firTab.d + (size_t)first * nTapCols : nullptr;      // ... and the FIR table
    if (ordered) CU(cudaStreamWaitEvent(stream, h->evLast, 0));          // stream-ordered after the instance's previous launch (see evLast)
    // the fused kernels run the canonical order; a plugin-order request may use them when the two orders provably agree
    const bool chainOrder = (h->period == 0 || pl.L.orderIndependent) && coreSel < 0 && !planOverride;
    int use = AVDSP_B200_KERNEL_GENERIC;
    if (chainOrder && h->kernelSel != AVDSP_B200_KERNEL_GENERIC) {
        if (h->kernelSel == AVDSP_B200_KERNEL_CHAIN_V1)
            return setErr(AVDSP_B200_ERR_UNSUPPORTED, "the first, tile-synchronous chain kernel was removed; use AVDSP_B200_KERNEL_CHAIN");
        if (pl.chain2Usable) use = AVDSP_B200_KERNEL_CHAIN;
    }
    // X/Y dataflow programs: the DAG kernel when no other fused kernel takes the program (or on request)
    if (chainOrder && pl.dagUsable && ((h->kernelSel == AVDSP_B200_KERNEL_AUTO && use == AVDSP_B200_KERNEL_GENERIC && !pl.mixUsable && !pl.firUsable) ||
                                        h->kernelSel == AVDSP_B200_KERNEL_DAG)) use = AVDSP_B200_KERNEL_DAG;
    if (h->kernelSel == AVDSP_B200_KERNEL_DAG && use != AVDSP_B200_KERNEL_DAG)
        return setErr(AVDSP_B200_ERR_UNSUPPORTED, "DAG kernel requested but this program/order does not map to it: " + pl.L.dagWhyNot);
    if (chainOrder && pl.mixUsable && (h->kernelSel == AVDSP_B200_KERNEL_AUTO || h->kernelSel == AVDSP_B200_KERNEL_MIX)) use = AVDSP_B200_KERNEL_MIX;
    if (chainOrder && pl.firUsable && (h->kernelSel == AVDSP_B200_KERNEL_AUTO || h->kernelSel == AVDSP_B200_KERNEL_FIR)) use = AVDSP_B200_KERNEL_FIR;
    // tensor-core Toeplitz GEMM: the bit-exact int8-limb form is the default for fixed-point batches that fill a tile;
    // the 3xTF32 form (stated tolerance) only on request.  With a per-stream FIR table the int8-limb form runs per stream (a
    // CTA = 128 outputs x 64 output blocks of one stream), which AUTO takes when a call fills those 64 blocks (8192 frames);
    // the 3xTF32 form takes shared taps only
    const bool fixedTc = pl.L.fir.aluClass == ALU_INT64 && pl.L.fir.maxLen >= 256;
    if (h->kernelSel == AVDSP_B200_KERNEL_FIR_TC && firTaps && pl.L.fir.aluClass != ALU_INT64)
        return setErr(AVDSP_B200_ERR_UNSUPPORTED, "the 3xTF32 tensor-core FIR kernel takes taps every stream shares; this instance has a per-stream FIR table");
    if (chainOrder && pl.firUsable && (h->kernelSel == AVDSP_B200_KERNEL_FIR_TC ||
        (h->kernelSel == AVDSP_B200_KERNEL_AUTO && fixedTc && (firTaps ? nFrames >= 8192 && !h->firTcPerFailed : n >= 32 && nFrames >= 128))))
        use = AVDSP_B200_KERNEL_FIR_TC;
    if (use == AVDSP_B200_KERNEL_FIR_TC && firTaps && !h->dFirTcPer && !h->firTcPerFailed) {
        // every stream's Toeplitz planes (C4: 4.3 MB per stream); when they do not fit, this instance runs k_fir with its table
        const size_t bytes = firTcPerTapsBytes(h->L.fir, h->nStreams);
        if (cudaMalloc(&h->dFirTcPer, bytes) != cudaSuccess) {
            cudaGetLastError();
            h->dFirTcPer = nullptr; h->firTcPerFailed = true;
            char line[160];
            snprintf(line, sizeof line, "per-stream tensor-core FIR: %zu MB of Toeplitz planes could not be allocated, k_fir runs the FIR table\n", bytes >> 20);
            h->trace += line;
        }
        h->firTcPerValid = false;
    }
    if (use == AVDSP_B200_KERNEL_FIR_TC && firTaps && h->firTcPerFailed) use = AVDSP_B200_KERNEL_FIR;
    if (h->kernelSel == AVDSP_B200_KERNEL_FIR_TC && use != AVDSP_B200_KERNEL_FIR_TC && !(firTaps && h->firTcPerFailed))
        return setErr(AVDSP_B200_ERR_UNSUPPORTED, "tensor-core FIR kernel requested but this program/order does not map to it: " + pl.L.firWhyNot);
    if (h->kernelSel == AVDSP_B200_KERNEL_FIR && use != AVDSP_B200_KERNEL_FIR)
        return setErr(AVDSP_B200_ERR_UNSUPPORTED, "FIR kernel requested but this program/order does not map to it: " + pl.L.firWhyNot);
    if (h->kernelSel == AVDSP_B200_KERNEL_MIX && use != AVDSP_B200_KERNEL_MIX)
        return setErr(AVDSP_B200_ERR_UNSUPPORTED, "mix kernel requested but the program has biquads or does not map to independent paths");
    if ((h->kernelSel == AVDSP_B200_KERNEL_CHAIN || h->kernelSel == AVDSP_B200_KERNEL_CHAIN_V1 || h->kernelSel == AVDSP_B200_KERNEL_CHAIN_V2 ||
         h->kernelSel == AVDSP_B200_KERNEL_CHAIN_V3) && use == AVDSP_B200_KERNEL_GENERIC)
        return setErr(AVDSP_B200_ERR_UNSUPPORTED, "chain kernel requested but this program/order does not map to it: " + pl.L.chainWhyNot);
    cudaError_t e;
    if (use == AVDSP_B200_KERNEL_FIR || use == AVDSP_B200_KERNEL_FIR_TC) {
        FirArgs A{};
        A.in = in; A.out = out; A.state = st; A.bigPool = pl.dBig;
        A.nStreams = n; A.nFrames = nFrames;
        A.inStreamStride = inSS; A.outStreamStride = outSS;
        A.inFrameStride = inFS; A.inChStride = inCS; A.outFrameStride = outFS; A.outChStride = outCS;
        int nl = 0;
        if (use == AVDSP_B200_KERNEL_FIR_TC && firTaps) {
            if (!h->firTcPerValid) {                              // rows changed since the planes were built: all streams again
                e = launchFirTcBuildTaps(h->L.fir, h->firTab.d, nTapCols, h->nStreams, h->dFirTcPer, stream);
                if (e != cudaSuccess) return cudaErr(e, "kernel launch");
                h->firTcPerValid = true;
                h->launches++;
            }
            const size_t need = firTcPerWorkspaceBytes(pl.L.fir, n, nFrames);
            if (need > h->firWsBytes) {
                CU(cudaStreamSynchronize(stream));
                if (h->dFirWs) cudaFree(h->dFirWs);
                h->dFirWs = nullptr; h->firWsBytes = 0;
                CU(cudaMalloc(&h->dFirWs, need));
                h->firWsBytes = need;
            }
            A.taps = firTaps; A.tapPitch = nTapCols;
            e = launchFirTcPer(pl.L.fir, A, h->dFirTcPer + (size_t)first * (firTcPerTapsBytes(h->L.fir, 1)), h->dFirWs, stream, &nl);
        } else if (use == AVDSP_B200_KERNEL_FIR_TC) {
            const int kind = pl.L.fir.aluClass == ALU_INT64 ? FIRTC_I8 : FIRTC_TF32;
            const size_t need = firTcWorkspaceBytes(pl.L.fir, kind, n, nFrames);
            if (need > h->firWsBytes) {
                CU(cudaStreamSynchronize(stream));
                if (h->dFirWs) cudaFree(h->dFirWs);
                h->dFirWs = nullptr; h->firWsBytes = 0;
                CU(cudaMalloc(&h->dFirWs, need));
                h->firWsBytes = need;
            }
            e = launchFirTc(pl.L.fir, kind, A, pl.dFirTaps, h->dFirWs, stream, &nl);
        } else {
            A.taps = firTaps; A.tapPitch = nTapCols;
            A.skip = firTaps && pl.L.fir.aluClass == ALU_F32 ? h->dFirFlags + first : nullptr;
            e = launchFir(pl.L.fir, A, h->numSMs, stream, &nl);
            if (e == cudaSuccess && A.skip) {
                // float rows with a tap the FIR kernels cannot multiply exactly: their CTAs did nothing, and the interpreter
                // runs those streams now from their untouched state blocks (one launch; streams without the flag return at once)
                GenericArgs X{};
                X.in = in; X.out = out; X.state = st; X.bigPool = pl.dBig;
                X.nStreams = n; X.nFrames = nFrames;
                X.inStreamStride = inSS; X.outStreamStride = outSS;
                X.inFrameStride = inFS; X.inChStride = inCS; X.outFrameStride = outFS; X.outChStride = outCS;
                X.coreSel = -1; X.period = 0;
                X.redo = A.skip; X.snapshot = st;
                X.coefs = coefs; X.coefPitch = h->nStreams; X.coefStep = 5 * pl.L.nFreq;
                X.firTaps = firTaps; X.firPitch = nTapCols; X.firCol = pl.dFirCol;
                for (int c = 0; c < P.nCores && c < kMaxCores; c++) { X.coreInMask[c] = pl.L.cores[c].usedIn; X.coreOutMask[c] = pl.L.cores[c].usedOut; }
                e = launchGeneric(G, X, stream);
                nl++;
            }
        }
        h->lastKernel = use;
        h->launches += nl - 1;
    } else if (use == AVDSP_B200_KERNEL_MIX) {
        MixArgs A{};
        A.in = in; A.out = out; A.state = st;
        A.nStreams = n; A.nFrames = nFrames;
        A.inStreamStride = inSS; A.outStreamStride = outSS;
        A.inFrameStride = inFS; A.inChStride = inCS; A.outFrameStride = outFS; A.outChStride = outCS;
        A.vecIn = inCS == 1 && inFS == nIn && (inSS & 3) == 0 && ((size_t)in & 15) == 0;
        A.vecOut = outCS == 1 && (nOut & 3) == 0 && (outFS & 3) == 0 && (outSS & 3) == 0 && ((size_t)out & 15) == 0;
        int J = 1, Lseg = nFrames;
        mixPrngSegments(pl.mix, A, h->numSMs, &J, &Lseg);
        if (pl.mix.hasCalc || pl.mix.anyTpdf) {
            const size_t need = (size_t)n * nFrames;
            if (need > h->tpdfWords) { if (h->dTpdf) cudaFree(h->dTpdf); h->dTpdf = nullptr; CU(cudaMalloc(&h->dTpdf, need * 4)); h->tpdfWords = need; }
            constexpr int kJumpLevels = kMixJumpLevels;       // thread j applies M^(2L * 2^b) for the bits b set in j
            if (!h->dJump) CU(cudaMalloc(&h->dJump, kJumpLevels * 128 * 4 * sizeof(unsigned)));
            if (h->jumpL != Lseg) {
                std::vector<unsigned> m(kJumpLevels * 128 * 4);
                for (int b = 0; b < kJumpLevels; b++) mixJumpMatrix((2ll * Lseg) << b, m.data() + b * 128 * 4);   // one TPDF value = two xoshiro128+ steps
                CU(cudaMemcpyAsync(h->dJump, m.data(), m.size() * 4, cudaMemcpyHostToDevice, stream));
                CU(cudaStreamSynchronize(stream));
                h->jumpL = Lseg;
            }
        }
        A.tpdfBuf = h->dTpdf;
        int nl = 1;
        e = launchMix(pl.mix, A, h->dJump, J, Lseg, h->numSMs, stream, &nl);
        h->lastKernel = AVDSP_B200_KERNEL_MIX;
        h->launches += nl - 1;                               // one is counted below
    } else if (use == AVDSP_B200_KERNEL_DAG) {
        Chain2Args A{};
        A.in = in; A.out = out; A.state = st; A.lanes = nullptr;
        A.nStreams = n; A.nFrames = nFrames;
        A.inStreamStride = inSS; A.outStreamStride = outSS;
        A.inFrameStride = inFS; A.inChStride = inCS; A.outFrameStride = outFS; A.outChStride = outCS;
        A.coefs = coefs; A.coefPitch = h->nStreams;
        e = launchDag(*pl.L.dag, pl.geomDag, A, stream);
        h->lastKernel = AVDSP_B200_KERNEL_DAG;
    } else if (use == AVDSP_B200_KERNEL_CHAIN) {
        Chain2Args A{};
        A.in = in; A.out = out; A.state = st; A.lanes = pl.dLanes2;
        A.nStreams = n; A.nFrames = nFrames;
        A.inStreamStride = inSS; A.outStreamStride = outSS;
        A.inFrameStride = inFS; A.inChStride = inCS; A.outFrameStride = outFS; A.outChStride = outCS;
        A.coefs = coefs; A.coefPitch = h->nStreams;
        // v3 (a cascade part per lane, lane = stream) wants full warps and several equal warps per sub-partition: AUTO takes it at
        // batch width (>= 16 streams per SM) when the cascades could be cut into parts of <= 4 sections (measured on C2: 9.06 ms
        // against v2's 9.50; with whole 6- and 8-section cascades per warp v3 is the slower one) and the call is long enough to
        // pay for v3's pipeline fill and drain (parts run a tile behind each other: C2 breaks even near 1500 frames per call --
        // 128 frames: v2 0.083 ms / v3 0.117, 1024: 0.262 / 0.267, 4096: 0.864 / 0.816); everything else runs on v2
        const bool v3Ok = pl.chain3Usable && use == AVDSP_B200_KERNEL_CHAIN;
        static const int envChain3 = [] { const char* v = getenv("AVDSP_B200_CHAIN3"); return (v && *v) ? atoi(v) : -1; }();
        bool v3 = v3Ok && h->kernelSel != AVDSP_B200_KERNEL_CHAIN_V2 &&
                  (h->kernelSel == AVDSP_B200_KERNEL_CHAIN_V3 || envChain3 == 1 ||
                   (envChain3 != 0 && pl.geom3.maxSec <= 4 && pl.geom3.streamsPerCta >= 16 && nFrames >= std::max(1536, 32 * pl.geom3.gmax)));
        if (h->kernelSel == AVDSP_B200_KERNEL_CHAIN_V3 && !v3)
            return setErr(AVDSP_B200_ERR_UNSUPPORTED, "chain kernel v3 requested but the program shape does not map to it");
        const bool flt = pl.L.chain.h.aluClass == ALU_F32;
        if (flt) {
            // the float class is the reference's arithmetic except next to the underflow threshold and beyond the binary32 range
            // (avdsp_dev.cuh, fltGuard): snapshot the state, let the cascades flag the streams that came near either, then list
            // the flagged streams, put their state back and run them again through k_chain2's exact form (hardware product +
            // integer fallback, the host's NaN rules).  Costs one state copy and two small launches when nothing is flagged.
            if (!h->dRedo) {
                CU(cudaMalloc(&h->dRedo, (size_t)h->nStreams * sizeof(int)));
                CU(cudaMalloc(&h->dRedoList, (size_t)h->nStreams * sizeof(int)));
                CU(cudaMalloc(&h->dRedoCount, (size_t)h->nStreams * sizeof(int)));       // one counter per run start (disjoint runs)
                CU(cudaMalloc(&h->dSnap, (size_t)h->nStreams * P.stateWords * sizeof(int)));
            }
            e = launchRedoPrepare(st, h->dSnap + (size_t)first * P.stateWords, (size_t)n * P.stateWords, h->dRedo + first, n, h->dRedoCount + first, stream);
            if (e != cudaSuccess) return cudaErr(e, "kernel launch");
            A.redo = h->dRedo + first;
        }
        if (v3) e = launchChain3(pl.L.chain, pl.geom3, A, stream);
        else e = launchChain2(pl.L.chain, pl.geom2, A, stream);
        if (flt && e == cudaSuccess) {
            e = launchRedoCompact(h->dRedo + first, n, h->dRedoList + first, h->dRedoCount + first, st, h->dSnap + (size_t)first * P.stateWords, P.stateWords, stream);
            if (e == cudaSuccess) {
                Chain2Args X = A;
                X.lanes = pl.dLanes2; X.redo = nullptr;
                X.map = h->dRedoList + first; X.countPtr = h->dRedoCount + first; X.exact = 1;
                Chain2Geom gx = pl.geom2;
                gx.floatFast = 0;                                // sources through the restatement as well
                e = launchChain2(pl.L.chain, gx, X, stream);
            }
            h->launches += 3;
        }
        h->lastChainVariant = v3 ? 3 : 2;
        h->lastKernel = AVDSP_B200_KERNEL_CHAIN;
    } else {
        GenericArgs A{};
        A.in = in; A.out = out; A.state = st; A.bigPool = pl.dBig;
        A.nStreams = n; A.nFrames = nFrames;
        A.inStreamStride = inSS; A.outStreamStride = outSS;
        A.inFrameStride = inFS; A.inChStride = inCS; A.outFrameStride = outFS; A.outChStride = outCS;
        A.coreSel = coreSel; A.period = coreSel >= 0 ? 0 : h->period;
        A.coefs = planOverride ? nullptr : coefs; A.coefPitch = h->nStreams; A.coefStep = 5 * pl.L.nFreq;
        A.firTaps = planOverride ? nullptr : firTaps; A.firPitch = nTapCols; A.firCol = pl.dFirCol;
        for (int c = 0; c < P.nCores && c < kMaxCores; c++) { A.coreInMask[c] = pl.L.cores[c].usedIn; A.coreOutMask[c] = pl.L.cores[c].usedOut; }
        e = launchGeneric(G, A, stream);
        h->lastKernel = AVDSP_B200_KERNEL_GENERIC;
    }
    if (e != cudaSuccess) return cudaErr(e, "kernel launch");
    if (ordered) CU(cudaEventRecord(h->evLast, stream));
    h->launches++;
    return 0;
}


// Streams [first, first+n): one launch, or one per run of streams that share a parameter variant.  The runs touch disjoint
// streams (state blocks, PCM rows), so they are launched on forked streams and joined: the kernels size a CTA for the whole
// batch, a run of a few streams is a few CTAs whatever it holds, and back to back on one stream every run would cost a whole
// launch's time.  Variants whose kernels share per-instance scratch (dither rows of the mix kernel, FIR workspace) stay in order.
static int launchRange(avdsp_b200* h, const int* in, int* out, int nFrames, int layout, int first, int n,
                       cudaStream_t stream, int coreSel = -1, const GenericPlan* planOverride = nullptr, int cap = 0) {
    if (h->variantOf.empty() || planOverride) return launchRun(h, *h, in, out, nFrames, layout, first, n, stream, coreSel, planOverride, cap);
    const PlanHeader& P = h->L.gen.h;
    const size_t c = (size_t)(cap > 0 ? cap : nFrames);
    bool fork = !(h->mixUsable || h->firUsable);
    for (const auto& v : h->variants) fork = fork && !(v->mixUsable || v->firUsable);
    int nRuns = 0;
    for (int a = first; a < first + n; nRuns++) { const int v = h->variantOf[a]; while (a < first + n && h->variantOf[a] == v) a++; }
    fork = fork && nRuns > 1;
    if (fork) {
        if (!h->evFork) {
            CU(cudaEventCreateWithFlags(&h->evFork, cudaEventDisableTiming));
            for (int k = 0; k < avdsp_b200::kVarStreams; k++) {
                CU(cudaStreamCreateWithFlags(&h->varStream[k], cudaStreamNonBlocking));
                CU(cudaEventCreateWithFlags(&h->varEv[k], cudaEventDisableTiming));
            }
        }
        CU(cudaStreamWaitEvent(stream, h->evLast, 0));
        CU(cudaEventRecord(h->evFork, stream));
    }
    int run = 0;
    for (int a = first; a < first + n; run++) {
        const int v = h->variantOf[a];
        int b = a + 1;
        while (b < first + n && h->variantOf[b] == v) b++;
        const size_t off = (size_t)(a - first) * c;                // both layouts are stream-major
        cudaStream_t s = stream;
        if (fork) {
            s = h->varStream[run % avdsp_b200::kVarStreams];
            if (run < avdsp_b200::kVarStreams) CU(cudaStreamWaitEvent(s, h->evFork, 0));
        }
        const int r = launchRun(h, v ? *h->variants[v - 1] : *h, in ? in + off * P.nIn : in, out ? out + off * P.nOut : out, nFrames, layout,
                                a, b - a, s, coreSel, nullptr, cap, !fork);
        if (r < 0) return r;
        a = b;
    }
    if (fork) {
        for (int k = 0; k < std::min(run, (int)avdsp_b200::kVarStreams); k++) {
            CU(cudaEventRecord(h->varEv[k], h->varStream[k]));
            CU(cudaStreamWaitEvent(stream, h->varEv[k], 0));
        }
        CU(cudaEventRecord(h->evLast, stream));
    }
    return 0;
}

// What follows a write of rows [first, first + n) of a table, on `s` after the write.  Only the FIR table has data derived from
// its rows: the per-stream Toeplitz planes are stale, and float programs recompute those streams' exactness flags.
static int rowsChanged(avdsp_b200* h, StreamTable avdsp_b200::* tab, int first, int n, cudaStream_t s) {
    if (tab != &avdsp_b200::firTab) return 0;
    h->firTcPerValid = false;
    if (h->L.gen.h.aluClass != ALU_F32) return 0;
    if (!h->dFirFlags) CU(cudaMalloc(&h->dFirFlags, (size_t)h->nStreams * 4));
    k_fir_tap_flags<<<(unsigned)((n + 7) / 8), 256, 0, s>>>(h->firTab.d, (int)h->L.firTapWords.size(), first, n, h->dFirFlags);
    CU(cudaGetLastError());
    h->launches++;
    return 0;
}

// host-side access to an instance's device data: after everything that was launched on it, on any stream
static int quiesce(avdsp_b200* h) {
    CU(cudaSetDevice(h->device));
    CU(cudaEventSynchronize(h->evLast));
    CU(cudaStreamSynchronize(h->stream));
    return 0;
}

static int ensureSlots(avdsp_b200* h, size_t inWords, size_t outWords) {
    for (int k = 0; k < avdsp_b200::kSlots; k++)
        if (!h->slotStream[k]) {
            CU(cudaStreamCreateWithFlags(&h->slotStream[k], cudaStreamNonBlocking));
            CU(cudaEventCreateWithFlags(&h->evIn[k], cudaEventDisableTiming));
            CU(cudaEventCreateWithFlags(&h->evKernel[k], cudaEventDisableTiming));
            CU(cudaEventCreateWithFlags(&h->evOut[k], cudaEventDisableTiming));
        }
    if (inWords > h->slotInWords) {
        for (int k = 0; k < avdsp_b200::kSlots; k++) { if (h->slotIn[k]) cudaFree(h->slotIn[k]); h->slotIn[k] = nullptr; }
        for (int k = 0; k < avdsp_b200::kSlots; k++) CU(cudaMalloc(&h->slotIn[k], inWords * 4));
        h->slotInWords = inWords;
    }
    if (outWords > h->slotOutWords) {
        for (int k = 0; k < avdsp_b200::kSlots; k++) { if (h->slotOut[k]) cudaFree(h->slotOut[k]); h->slotOut[k] = nullptr; }
        for (int k = 0; k < avdsp_b200::kSlots; k++) CU(cudaMalloc(&h->slotOut[k], outWords * 4));
        h->slotOutWords = outWords;
    }
    return 0;
}

extern "C" {

int avdsp_b200_process_range(avdsp_b200_t* h, const void* in, void* out, int nFrames, int layout,
                             int firstStream, int nStreams, void* cudaStream) {
    if (!h) return setErr(AVDSP_B200_ERR_ARG, "NULL instance");
    NO_MULTI(h, "avdsp_b200_process_range / _async");
    if (nFrames < 0 || firstStream < 0 || nStreams < 0 || firstStream + nStreams > h->nStreams) return setErr(AVDSP_B200_ERR_ARG, "bad frame/stream range");
    if ((!in && h->L.gen.h.nIn) || (!out && h->L.gen.h.nOut)) return setErr(AVDSP_B200_ERR_ARG, "NULL buffer");
    CU(cudaSetDevice(h->device));
    return launchRange(h, (const int*)in, (int*)out, nFrames, layout, firstStream, nStreams, (cudaStream_t)cudaStream);
}

int avdsp_b200_process_async(avdsp_b200_t* h, const void* in, void* out, int nFrames, int layout, void* cudaStream) {
    if (!h) return setErr(AVDSP_B200_ERR_ARG, "NULL instance");
    return avdsp_b200_process_range(h, in, out, nFrames, layout, 0, h->nStreams, cudaStream);
}

} // extern "C"

// host buffers of a single-device instance; copyOnly: the same DMA schedule without the launches (the copy roofline of the host path)
static int processHost(avdsp_b200* h, const void* in, void* out, int nFrames, int layout, bool copyOnly) {
    CU(cudaSetDevice(h->device));
    // Host buffers.  The time loop of a launch is sequential, so cutting the batch by streams would only shrink
    // the grid; the batch is cut in TIME instead: chunk c of every stream is copied in (one strided 2-D DMA),
    // processed by one launch over all streams, and copied out, through kSlots staging buffers.  Three CUDA
    // streams (copy-in, compute, copy-out) linked by events keep PCIe in both directions and the SMs busy at
    // once; launches stay in order on the compute stream because chunk c+1 continues chunk c's state.
    const PlanHeader& P = h->L.gen.h;
    if ((!in && P.nIn) || (!out && P.nOut)) return setErr(AVDSP_B200_ERR_ARG, "NULL buffer");
    const size_t S = (size_t)h->nStreams;
    const size_t perFrame = std::max<size_t>((size_t)(P.nIn + P.nOut) * S, 1);       // words per frame over all streams
    long long chunk = (long long)(((size_t)96 << 20) / perFrame);                     // ~384 MB of PCM per chunk
    chunk = std::max<long long>(256, chunk / 256 * 256);
    if (const char* ev = getenv("AVDSP_B200_HOST_CHUNK")) { const long long v = atoll(ev); if (v > 0) chunk = v; }   // tests: force several chunks
    if (chunk > nFrames) chunk = nFrames;
    const int r0 = ensureSlots(h, std::max<size_t>(S * chunk * P.nIn, 1), std::max<size_t>(S * chunk * P.nOut, 1));
    if (r0 < 0) return r0;
    cudaStream_t sIn = h->slotStream[0], sK = h->slotStream[1], sOut = h->slotStream[2];
    const int32_t* hin = (const int32_t*)in; int32_t* hout = (int32_t*)out;
    // rows of the 2-D copies: one per stream (interleaved) or per (stream, channel) (planar)
    const bool il = layout == AVDSP_B200_INTERLEAVED;
    if (!il && layout != AVDSP_B200_PLANAR) return setErr(AVDSP_B200_ERR_ARG, "unknown layout");
    const size_t inRows = il ? S : S * P.nIn, outRows = il ? S : S * P.nOut;
    const size_t inRowW = il ? P.nIn : 1, outRowW = il ? P.nOut : 1;                   // words per frame inside a row
    int slot = 0;
    for (long long f0 = 0; f0 < nFrames; f0 += chunk, slot = (slot + 1) % avdsp_b200::kSlots) {
        const int nf = (int)std::min<long long>(chunk, nFrames - f0);
        // slot reuse: the copy-in may overwrite slotIn only after the launch that read it, and the launch may overwrite
        // slotOut only after its copy-out
        CU(cudaStreamWaitEvent(sIn, h->evKernel[slot], 0));
        if (P.nIn)
            CU(cudaMemcpy2DAsync(h->slotIn[slot], (size_t)chunk * inRowW * 4, hin + (size_t)f0 * inRowW, (size_t)nFrames * inRowW * 4,
                                 (size_t)nf * inRowW * 4, inRows, cudaMemcpyHostToDevice, sIn));
        CU(cudaEventRecord(h->evIn[slot], sIn));
        CU(cudaStreamWaitEvent(sK, h->evIn[slot], 0));
        CU(cudaStreamWaitEvent(sK, h->evOut[slot], 0));
        if (!copyOnly) {
            const int r = launchRange(h, h->slotIn[slot], h->slotOut[slot], nf, layout, 0, h->nStreams, sK, -1, nullptr, (int)chunk);
            if (r < 0) return r;
        }
        CU(cudaEventRecord(h->evKernel[slot], sK));
        CU(cudaStreamWaitEvent(sOut, h->evKernel[slot], 0));
        if (P.nOut)
            CU(cudaMemcpy2DAsync(hout + (size_t)f0 * outRowW, (size_t)nFrames * outRowW * 4, h->slotOut[slot], (size_t)chunk * outRowW * 4,
                                 (size_t)nf * outRowW * 4, outRows, cudaMemcpyDeviceToHost, sOut));
        CU(cudaEventRecord(h->evOut[slot], sOut));
    }
    CU(cudaStreamSynchronize(sOut));
    CU(cudaStreamSynchronize(sK));
    CU(cudaStreamSynchronize(sIn));
    return 0;
}


// ---- multi-device instances: fan a call out over the shards, one host thread per GPU running next to it ----
template <typename Fn>
static int forShards(avdsp_b200* h, Fn fn) {
    const size_t n = h->shards.size();
    std::vector<int> rc(n, 0);
    std::vector<std::string> msg(n);
    std::vector<std::thread> th;
    th.reserve(n);
    for (size_t k = 0; k < n; k++)
        th.emplace_back([&, k] {
            if (h->shards[k]) bindThreadToNode(h->shards[k]->numaNode);      // staging thread next to its GPU (no-op when the topology is unknown)
            rc[k] = fn((int)k, h->shards[k]);
            if (rc[k] < 0) msg[k] = g_lastError;             // thread-local: carry it over to the caller's thread
        });
    for (auto& t : th) t.join();
    for (size_t k = 0; k < n; k++) if (rc[k] < 0) return setErr(rc[k], "device " + std::to_string(h->shards[k]->device) + ": " + msg[k]);
    return 0;
}
static int shardOf(const avdsp_b200* h, int stream) {
    int k = 0;
    while (k + 1 < (int)h->shards.size() && stream >= h->shardFirst[k + 1]) k++;
    return k;
}
static int resetShards(avdsp_b200* h, int fs, const int32_t* seeds, int defaultDither) {
    if (fs != h->L.fs || defaultDither != h->L.defaultDither) {
        Lowered nl;
        const int rc = decodeAt(*h, fs, defaultDither, &nl); if (rc < 0) return rc;
        h->L = std::move(nl);
    }
    if (seeds) h->seeds.assign(seeds, seeds + h->nStreams); else h->seeds.clear();
    return forShards(h, [&](int k, avdsp_b200* sh) { return avdsp_b200_reset(sh, fs, seeds ? seeds + h->shardFirst[k] : nullptr, defaultDither); });
}

extern "C" {

int avdsp_b200_process(avdsp_b200_t* h, const void* in, void* out, int nFrames, int layout, int memspace) {
    if (!h) return setErr(AVDSP_B200_ERR_ARG, "NULL instance");
    if (nFrames < 0) return setErr(AVDSP_B200_ERR_ARG, "negative frame count");
    if (nFrames == 0) return 0;
    if (!h->shards.empty()) {
        if (memspace != AVDSP_B200_HOST) return setErr(AVDSP_B200_ERR_UNSUPPORTED, "a multi-device instance processes HOST buffers (device buffers belong to one GPU)");
        if (layout != AVDSP_B200_INTERLEAVED && layout != AVDSP_B200_PLANAR) return setErr(AVDSP_B200_ERR_ARG, "unknown layout");
        const PlanHeader& P = h->L.gen.h;
        // both layouts are stream-major: shard k's streams are one contiguous slice of either buffer
        return forShards(h, [&](int k, avdsp_b200* sh) {
            const size_t f = (size_t)h->shardFirst[k] * (size_t)nFrames;
            return avdsp_b200_process(sh, (const int32_t*)in + f * P.nIn, (int32_t*)out + f * P.nOut, nFrames, layout, AVDSP_B200_HOST);
        });
    }
    CU(cudaSetDevice(h->device));
    if (memspace == AVDSP_B200_DEVICE) {
        const int r = avdsp_b200_process_range(h, in, out, nFrames, layout, 0, h->nStreams, h->stream);
        if (r < 0) return r;
        CU(cudaStreamSynchronize(h->stream));
        return 0;
    }
    if (memspace != AVDSP_B200_HOST) return setErr(AVDSP_B200_ERR_ARG, "unknown memspace");
    return processHost(h, in, out, nFrames, layout, false);
}

int avdsp_b200_copy_only(avdsp_b200_t* h, const void* in, void* out, int nFrames, int layout) {
    if (!h) return setErr(AVDSP_B200_ERR_ARG, "NULL instance");
    if (nFrames <= 0) return nFrames < 0 ? setErr(AVDSP_B200_ERR_ARG, "negative frame count") : 0;
    if (!h->shards.empty()) {
        const PlanHeader& P = h->L.gen.h;
        return forShards(h, [&](int k, avdsp_b200* sh) {
            const size_t f = (size_t)h->shardFirst[k] * (size_t)nFrames;
            return avdsp_b200_copy_only(sh, (const int32_t*)in + f * P.nIn, (int32_t*)out + f * P.nOut, nFrames, layout);
        });
    }
    return processHost(h, in, out, nFrames, layout, true);
}

int avdsp_b200_create_multi(avdsp_b200_t** out, const int32_t* prog, int progWords, int fs, int format,
                            int nStreams, const int32_t* seeds, int defaultDither, unsigned deviceMask) {
    if (!out) return setErr(AVDSP_B200_ERR_ARG, "out is NULL");
    *out = nullptr;
    if (nStreams < 1) return setErr(AVDSP_B200_ERR_ARG, "nStreams must be >= 1");
    std::unique_ptr<avdsp_b200, void (*)(avdsp_b200*)> h(new avdsp_b200, freeAll);
    std::string err;
    const int rc = decodeProgram(prog, progWords, 0x7FFFFFFF, format, fs, defaultDither, &h->L, &err);
    if (rc < 0) return setErr(rc, err);
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return setErr(AVDSP_B200_ERR_CUDA, std::string("no CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0") +
                                               " (avdsp_b200 has no CPU fallback)");
    std::vector<int> devs;
    for (int d = 0; d < 32; d++) if ((deviceMask >> d) & 1u) { if (d >= ndev) return setErr(AVDSP_B200_ERR_ARG, "deviceMask names a device that does not exist"); devs.push_back(d); }
    if (devs.empty()) return setErr(AVDSP_B200_ERR_ARG, "deviceMask is empty");
    if (const char* rp = getenv("AVDSP_B200_MULTI_REPLICATE")) {       // tests on a one-GPU box: every device of the mask carries k shards
        const int k = atoi(rp);
        if (k > 1 && k <= 16) { const std::vector<int> base = devs; for (int i = 1; i < k; i++) devs.insert(devs.end(), base.begin(), base.end()); }
    }
    if ((int)devs.size() > nStreams) devs.resize(nStreams);
    h->device = -1; h->nStreams = nStreams;
    if (seeds) h->seeds.assign(seeds, seeds + nStreams);
    // contiguous balanced ranges, the first (nStreams mod n) shards one stream longer (avdsp_b200/sharding.py: same partition)
    const int n = (int)devs.size(), q = nStreams / n, r = nStreams % n;
    h->shardFirst.assign(1, 0);
    for (int k = 0; k < n; k++) h->shardFirst.push_back(h->shardFirst.back() + q + (k < r ? 1 : 0));
    h->shards.assign(n, nullptr);
    const int frc = forShards(h.get(), [&](int k, avdsp_b200* /*not created yet*/) {
        const int first = h->shardFirst[k], cnt = h->shardFirst[k + 1] - first;
        char bus[64] = {0};
        if (cudaDeviceGetPCIBusId(bus, sizeof bus, devs[k]) == cudaSuccess) bindThreadToNode(numaNodeOfPci(bus));   // state and staging allocations next to the GPU
        return std::min(0, avdsp_b200_create(&h->shards[k], prog, progWords, fs, format, cnt, seeds ? seeds + first : nullptr, defaultDither, devs[k]));
    });
    if (frc < 0) { for (auto& sh : h->shards) { if (sh) freeAll(sh); } h->shards.clear(); return frc; }
    h->trace = h->shards[0]->trace;
    h->numSMs = h->shards[0]->numSMs;
    g_lastError.clear();
    *out = h.release();
    return rc;
}

int avdsp_b200_num_devices(const avdsp_b200_t* h) { return !h ? 0 : h->shards.empty() ? 1 : (int)h->shards.size(); }
int avdsp_b200_shard_info(const avdsp_b200_t* h, int k, int* device, int* firstStream, int* nStreams, int* numaNode) {
    if (!h || k < 0 || k >= avdsp_b200_num_devices(h)) return setErr(AVDSP_B200_ERR_ARG, "bad shard index");
    const avdsp_b200* sh = h->shards.empty() ? h : h->shards[k];
    if (device) *device = sh->device;
    if (firstStream) *firstStream = h->shards.empty() ? 0 : h->shardFirst[k];
    if (nStreams) *nStreams = sh->nStreams;
    if (numaNode) *numaNode = sh->numaNode;
    return 0;
}

// PCM buffers placed for the instance: page-locked, and every shard's slice ([stream][...] layouts: contiguous) on the host
// NUMA node next to the GPU that will DMA it.  bytesPerStream = nFrames * channels * 4 for the buffer in question.
void* avdsp_b200_host_alloc(avdsp_b200_t* h, size_t bytesPerStream) {
    if (!h || bytesPerStream == 0) { setErr(AVDSP_B200_ERR_ARG, "bad argument"); return nullptr; }
    const int n = avdsp_b200_num_devices(h);
    std::vector<size_t> off(1, 0);
    std::vector<int> nodes;
    for (int k = 0; k < n; k++) {
        int first = 0, cnt = 0, node = -1;
        avdsp_b200_shard_info(h, k, nullptr, &first, &cnt, &node);
        off.push_back((size_t)(first + cnt) * bytesPerStream);
        nodes.push_back(node);
    }
    const size_t bytes = (size_t)h->nStreams * bytesPerStream;
    void* p = hostAllocPlaced(bytes, off, nodes);
    if (!p) { setErr(AVDSP_B200_ERR_ARG, "host allocation failed"); return nullptr; }
    const cudaError_t e = cudaHostRegister(p, bytes, cudaHostRegisterPortable);
    if (e != cudaSuccess) { hostFreePlaced(p, bytes); cudaErr(e, "cudaHostRegister"); return nullptr; }
    h->hostAllocs[p] = bytes;
    return p;
}
void avdsp_b200_host_free(avdsp_b200_t* h, void* p) {
    if (!h || !p) return;
    auto it = h->hostAllocs.find(p);
    if (it == h->hostAllocs.end()) return;
    cudaHostUnregister(p);
    hostFreePlaced(p, it->second);
    h->hostAllocs.erase(it);
}

} // extern "C"

extern "C" {

int avdsp_b200_process_pcm(avdsp_b200_t* h, const void* in, int pcmFormat, void* out, int nFrames, int memspace) {
    if (!h) return setErr(AVDSP_B200_ERR_ARG, "NULL instance");
    if (pcmFormat == AVDSP_B200_PCM_S32) return avdsp_b200_process(h, in, out, nFrames, AVDSP_B200_INTERLEAVED, memspace);
    if (pcmFormat != AVDSP_B200_PCM_S16 && pcmFormat != AVDSP_B200_PCM_S24_3LE) return setErr(AVDSP_B200_ERR_ARG, "unknown PCM format");
    if (nFrames < 0) return setErr(AVDSP_B200_ERR_ARG, "negative frame count");
    if (nFrames == 0) return 0;
    if (!h->shards.empty()) {
        if (memspace != AVDSP_B200_HOST) return setErr(AVDSP_B200_ERR_UNSUPPORTED, "a multi-device instance processes HOST buffers");
        const PlanHeader& PP = h->L.gen.h;
        const size_t bps = pcmFormat == AVDSP_B200_PCM_S16 ? 2 : 3;
        return forShards(h, [&](int k, avdsp_b200* sh) {
            const size_t f = (size_t)h->shardFirst[k] * (size_t)nFrames;
            return avdsp_b200_process_pcm(sh, (const unsigned char*)in + f * PP.nIn * bps, pcmFormat, (int32_t*)out + f * PP.nOut, nFrames, memspace);
        });
    }
    CU(cudaSetDevice(h->device));
    const PlanHeader& P = h->L.gen.h;
    const size_t nIn = (size_t)h->nStreams * nFrames * P.nIn, nOut = (size_t)h->nStreams * nFrames * P.nOut;
    const size_t rawBytes = nIn * (pcmFormat == AVDSP_B200_PCM_S16 ? 2 : 3);
    if (nIn > h->pcmInWords) { if (h->pcmIn) cudaFree(h->pcmIn); h->pcmIn = nullptr; CU(cudaMalloc(&h->pcmIn, std::max<size_t>(nIn, 1) * 4)); h->pcmInWords = nIn; }
    const unsigned char* raw = (const unsigned char*)in;
    if (memspace == AVDSP_B200_HOST) {
        if (rawBytes > h->pcmRawBytes) { if (h->pcmRaw) cudaFree(h->pcmRaw); h->pcmRaw = nullptr; CU(cudaMalloc(&h->pcmRaw, std::max<size_t>(rawBytes, 1))); h->pcmRawBytes = rawBytes; }
        if (nOut > h->pcmOutWords) { if (h->pcmOut) cudaFree(h->pcmOut); h->pcmOut = nullptr; CU(cudaMalloc(&h->pcmOut, std::max<size_t>(nOut, 1) * 4)); h->pcmOutWords = nOut; }
        CU(cudaMemcpyAsync(h->pcmRaw, in, rawBytes, cudaMemcpyHostToDevice, h->stream));
        raw = (const unsigned char*)h->pcmRaw;
    } else if (memspace != AVDSP_B200_DEVICE) return setErr(AVDSP_B200_ERR_ARG, "unknown memspace");
    if (nIn) {
        k_widen_pcm<<<(unsigned)((nIn + 255) / 256), 256, 0, h->stream>>>(raw, pcmFormat, h->pcmIn, nIn);
        CU(cudaGetLastError());
        h->launches++;
    }
    int* dout = memspace == AVDSP_B200_HOST ? h->pcmOut : (int*)out;
    const int r = launchRange(h, h->pcmIn, dout, nFrames, AVDSP_B200_INTERLEAVED, 0, h->nStreams, h->stream);
    if (r < 0) return r;
    if (memspace == AVDSP_B200_HOST && nOut) CU(cudaMemcpyAsync(out, h->pcmOut, nOut * 4, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return 0;
}

} // extern "C"

// ---- per-stream parameter overrides (SURVEY.md 8f-3; the dump-file workflow per stream) -------------------------------
// plans for `words` (the loaded program with some PARAM words replaced): an existing variant with exactly these words, or a new one
static int variantFor(avdsp_b200* h, const std::vector<int32_t>& words, int* id) {
    if (words == h->L.words) { *id = 0; return 0; }
    for (size_t k = 0; k < h->variants.size(); k++) if (h->variants[k]->L.words == words) { *id = (int)k + 1; return 0; }
    std::unique_ptr<Plans> v(new Plans);
    v->L = h->L;
    std::string err;
    const int rc = relowerProgram(words.data(), (int)words.size(), &v->L, &err);       // same opcode structure, same state layout, else an error
    if (rc < 0) return setErr(rc, err);
    const int r = uploadPlanData(*v, h->device, h->nStreams, h->numSMs);
    if (r < 0) return r;
    h->variants.push_back(std::move(v));
    *id = (int)h->variants.size();
    return 0;
}

// ---- per-stream tables (StreamTable, instance.h): the biquad coefficient table and the FIR table ---------------------
// A table's column list for a program.  The list does not depend on the rate: lower at the lowest one the header admits
// (decodeProgram validates it).  allRates: the program must also lower at every other rate it admits, as describe would check
// each of them.
static int tableWords(std::vector<int32_t> Lowered::* list, bool allRates, const int32_t* prog, int progWords, int format,
                      int32_t* wordIndex, int maxOut) {
    if (maxOut < 0 || (maxOut > 0 && !wordIndex)) return setErr(AVDSP_B200_ERR_ARG, "bad output buffer");
    const int fi = (prog && progWords > H_FREQMIN) ? prog[H_FREQMIN] : 0;
    const int fs = (fi >= 0 && fi < kNumFreq) ? kFreqTable[fi] : 0;
    std::unique_ptr<Lowered> L(new Lowered);
    std::string err;
    int rc = decodeProgram(prog, progWords, 0x7FFFFFFF, format, fs, 31, L.get(), &err);
    if (rc < 0) return setErr(rc, err);
    if (allRates) {
        std::unique_ptr<Lowered> Lr(new Lowered);
        for (int f = fi + 1; f <= prog[H_FREQMAX] && f < kNumFreq; f++) {
            rc = decodeProgram(prog, progWords, 0x7FFFFFFF, format, kFreqTable[f], 31, Lr.get(), &err);
            if (rc < 0) return setErr(rc, err);
        }
    }
    const std::vector<int32_t>& w = (*L).*list;
    const int n = (int)w.size();
    for (int k = 0; k < n && k < maxOut; k++) wordIndex[k] = w[k];
    return n;
}

// A table, created on first use: every stream's row holds the words it runs with now (the program's, or its variant's).
// Synchronous: the table is not in use yet.
static int ensureTable(avdsp_b200* h, StreamTable avdsp_b200::* tab) {
    StreamTable& t = h->*tab;
    if (t.d) return 0;
    const std::vector<int32_t>& cols = h->L.*t.words;
    const size_t N = (size_t)h->nStreams, nc = cols.size(), ss = t.streamStride(nc), cs = t.colStride(N);
    std::vector<int32_t> init(nc * N);
    for (size_t s = 0; s < N; s++) {
        const int v = h->variantOf.empty() ? 0 : h->variantOf[s];
        const std::vector<int32_t>& w = v ? h->variants[v - 1]->L.words : h->L.words;
        for (size_t c = 0; c < nc; c++) init[s * ss + c * cs] = w[cols[c]];
    }
    int* d = nullptr;
    CU(cudaMalloc(&d, init.size() * 4));
    t.d = d;
    cudaError_t e = cudaMemcpyAsync(d, init.data(), init.size() * 4, cudaMemcpyHostToDevice, h->stream);
    int r = e == cudaSuccess ? rowsChanged(h, tab, 0, h->nStreams, h->stream) : cudaErr(e, "table upload");
    if (r >= 0 && (e = cudaStreamSynchronize(h->stream)) != cudaSuccess) r = cudaErr(e, "table upload");
    if (r < 0) { cudaFree(d); t.d = nullptr; }
    return r;
}

// Rows [nStreams][columns] for streams [firstStream, firstStream + nStreams) of a table, from HOST or DEVICE memory, in the
// instance's stream order.  refusal: why this program can have no such table (nullptr: it can).  A refused call changes nothing.
static int setRows(avdsp_b200* h, StreamTable avdsp_b200::* tab, const char* refusal, int firstStream, int nStreams,
                   const int32_t* values, int memspace, void* cudaStream) {
    if (!h || !values) return setErr(AVDSP_B200_ERR_ARG, "NULL argument");
    if (firstStream < 0 || nStreams < 0 || (long long)firstStream + nStreams > h->nStreams) return setErr(AVDSP_B200_ERR_ARG, "bad stream range");
    if (memspace != AVDSP_B200_HOST && memspace != AVDSP_B200_DEVICE) return setErr(AVDSP_B200_ERR_ARG, "unknown memspace");
    StreamTable& t = h->*tab;
    const std::vector<int32_t>& cols = h->L.*t.words;
    const int nCols = (int)cols.size();
    if (nCols == 0) return setErr(AVDSP_B200_ERR_UNSUPPORTED, std::string("the program has no ") + t.noun + " words");
    if (refusal) return setErr(AVDSP_B200_ERR_UNSUPPORTED, refusal);
    if (!h->shards.empty() && memspace != AVDSP_B200_HOST)
        return setErr(AVDSP_B200_ERR_UNSUPPORTED, std::string("a multi-device instance takes HOST ") + t.noun + " rows (device buffers belong to one GPU)");
    for (const avdsp_b200* o : h->shards.empty() ? std::vector<avdsp_b200*>{h} : h->shards)
        for (const auto& v : o->variants)
            if (v->L.*t.words != cols) return setErr(AVDSP_B200_ERR_UNSUPPORTED, std::string("a parameter variant moved the ") + t.noun + " words");
    if (!h->shards.empty())
        return forShards(h, [&](int k, avdsp_b200* sh) {
            const int a = std::max(firstStream, h->shardFirst[k]), b = std::min(firstStream + nStreams, h->shardFirst[k + 1]);
            if (b <= a) return 0;
            return setRows(sh, tab, refusal, a - h->shardFirst[k], b - a, values + (size_t)(a - firstStream) * nCols, AVDSP_B200_HOST, nullptr);
        });
    if (nStreams == 0) return 0;
    CU(cudaSetDevice(h->device));
    { const int r = ensureTable(h, tab); if (r < 0) return r; }
    const cudaStream_t s = memspace == AVDSP_B200_DEVICE ? (cudaStream_t)cudaStream : h->stream;
    const size_t words = (size_t)nStreams * nCols;
    CU(cudaStreamWaitEvent(s, h->evLast, 0));                 // after every launch enqueued on the instance before this call
    if (t.streamMajor) {                                      // rows arrive in the table's own layout: one copy
        CU(cudaMemcpyAsync(t.d + (size_t)firstStream * nCols, values, words * 4,
                           memspace == AVDSP_B200_HOST ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice, s));
    } else {
        const int* rows = values;
        if (memspace == AVDSP_B200_HOST) {
            if (words > t.stageWords) {
                CU(cudaStreamSynchronize(s));
                if (t.dStage) cudaFree(t.dStage);
                t.dStage = nullptr; t.stageWords = 0;
                CU(cudaMalloc(&t.dStage, words * 4));
                t.stageWords = words;
            }
            CU(cudaMemcpyAsync(t.dStage, values, words * 4, cudaMemcpyHostToDevice, s));
            rows = t.dStage;
        }
        k_coef_scatter<<<dim3((unsigned)((nStreams + 31) / 32), (unsigned)((nCols + 31) / 32)), dim3(32, 8), 0, s>>>(t.d, h->nStreams, firstStream, nStreams, nCols, rows);
        CU(cudaGetLastError());
        h->launches++;
    }
    { const int r = rowsChanged(h, tab, firstStream, nStreams, s); if (r < 0) return r; }
    CU(cudaEventRecord(h->evLast, s));
    if (memspace == AVDSP_B200_HOST) CU(cudaStreamSynchronize(s));    // the caller's buffer (and the staging rows) are free again
    return 0;
}

extern "C" {

int avdsp_b200_param_index(const avdsp_b200_t* h, int offset, int paramNum) {
    if (!h) return setErr(AVDSP_B200_ERR_ARG, "NULL instance");
    const std::vector<int32_t>& w = h->L.words;
    const int total = h->L.totalLength;
    if (paramNum == 0) return (offset >= 0 && offset < total) ? offset : setErr(AVDSP_B200_ERR_ARG, "parameter offset outside the program");
    // encoder/dsp_encoder.c:380-412 (findInParamSpace): relative to the first data word of the DSP_PARAM_NUM section with this number
    for (int p = 0; p < total;) {
        const int op = wordOpcode(w[p]), sk = wordSkip(w[p]);
        if (sk == 0) break;
        if (op == OP_PARAM_NUM && p + 1 < total && w[p + 1] == paramNum) {
            const int idx = p + 2 + offset;
            return (offset >= 0 && idx < p + sk) ? idx : setErr(AVDSP_B200_ERR_ARG, "parameter offset outside its DSP_PARAM_NUM section");
        }
        p += sk;
    }
    return setErr(AVDSP_B200_ERR_ARG, "no DSP_PARAM_NUM section with this number");
}

int avdsp_b200_set_param(avdsp_b200_t* h, int firstStream, int nStreams, int wordIndex, const int32_t* values, int nWords) {
    if (!h || !values) return setErr(AVDSP_B200_ERR_ARG, "NULL argument");
    if (firstStream < 0 || nStreams < 0 || firstStream + nStreams > h->nStreams) return setErr(AVDSP_B200_ERR_ARG, "bad stream range");
    if (wordIndex < 0 || nWords < 0 || wordIndex + nWords > h->L.totalLength) return setErr(AVDSP_B200_ERR_ARG, "parameter words outside the program");
    if (nStreams == 0 || nWords == 0) return 0;
    if (!h->shards.empty()) {
        for (size_t k = 0; k < h->shards.size(); k++) {
            const int a = std::max(firstStream, h->shardFirst[k]), b = std::min(firstStream + nStreams, h->shardFirst[k + 1]);
            if (b <= a) continue;
            const int r = avdsp_b200_set_param(h->shards[k], a - h->shardFirst[k], b - a, wordIndex, values, nWords);
            if (r < 0) return r;
        }
        return 0;
    }
    { const int q = quiesce(h); if (q < 0) return q; }
    // while the instance has a table, the words it holds are written into the streams' rows; the other words make variants as
    // without one.  Everything that can fail (lowering a variant) happens before anything changes.
    const decltype(&avdsp_b200::coefTab) tables[] = {&avdsp_b200::coefTab, &avdsp_b200::firTab};
    std::vector<int> colOf[2];                // table column of word k of the call, or -1
    std::vector<char> tableWord(nWords, 0);
    for (int t = 0; t < 2; t++) {
        colOf[t].assign(nWords, -1);
        if (!(h->*tables[t]).d) continue;
        const std::vector<int32_t>& list = h->L.*(h->*tables[t]).words;
        for (int k = 0; k < nWords; k++) {
            const auto it = std::lower_bound(list.begin(), list.end(), wordIndex + k);
            if (it != list.end() && *it == wordIndex + k) { colOf[t][k] = (int)(it - list.begin()); tableWord[k] = 1; }
        }
    }
    const bool anyVariantWord = std::count(tableWord.begin(), tableWord.end(), 0) > 0;
    // streams of the range may sit on different variants already: patch each of those once
    std::map<int, int> moved;                 // old variant -> new variant
    if (anyVariantWord) {
        const size_t nBefore = h->variants.size();
        auto undo = [&](int rc) { h->variants.resize(nBefore); return rc; };    // release the variants this call created; nothing else has changed yet
        for (int s = firstStream; s < firstStream + nStreams; s++) {
            const int old = h->variantOf.empty() ? 0 : h->variantOf[s];
            if (moved.count(old)) continue;
            std::vector<int32_t> words = old ? h->variants[old - 1]->L.words : h->L.words;
            for (int k = 0; k < nWords; k++) if (!tableWord[k]) words[wordIndex + k] = values[k];
            int id = 0;
            const int r = variantFor(h, words, &id);
            if (r < 0) return undo(r);
            for (auto tab : tables) {
                const StreamTable& t = h->*tab;
                if (t.d && id > 0 && h->variants[id - 1]->L.*t.words != h->L.*t.words)
                    return undo(setErr(AVDSP_B200_ERR_UNSUPPORTED, std::string("this change moves ") + t.noun + " words the table holds"));
            }
            moved.emplace(old, id);
        }
    }
    for (int t = 0; t < 2; t++) {
        StreamTable& tab = h->*tables[t];
        if (!tab.d) continue;
        const size_t ss = tab.streamStride((h->L.*tab.words).size()), cs = tab.colStride(h->nStreams);
        bool any = false;
        std::vector<int32_t> col((size_t)nStreams);
        for (int k = 0; k < nWords; k++) {
            if (colOf[t][k] < 0) continue;
            std::fill(col.begin(), col.end(), values[k]);       // one word of every row of the range
            CU(cudaMemcpy2DAsync(tab.d + firstStream * ss + colOf[t][k] * cs, ss * 4, col.data(), 4, 4, (size_t)nStreams,
                                 cudaMemcpyHostToDevice, h->stream));
            CU(cudaStreamSynchronize(h->stream));
            any = true;
        }
        if (any) { const int r = rowsChanged(h, tables[t], firstStream, nStreams, h->stream); if (r < 0) return r; }
        CU(cudaEventRecord(h->evLast, h->stream));
    }
    if (!anyVariantWord) return 0;
    if (h->variantOf.empty()) h->variantOf.assign(h->nStreams, 0);
    for (int s = firstStream; s < firstStream + nStreams; s++) h->variantOf[s] = moved.at(h->variantOf[s]);
    // variants nobody runs any more are released (ids above shift down)
    std::vector<int> used(h->variants.size() + 1, 0);
    for (int v : h->variantOf) used[v] = 1;
    std::vector<int> remap(h->variants.size() + 1, 0);
    std::vector<std::unique_ptr<Plans>> keep;
    for (size_t k = 0; k < h->variants.size(); k++)
        if (used[k + 1]) { keep.push_back(std::move(h->variants[k])); remap[k + 1] = (int)keep.size(); }
    h->variants.swap(keep);
    bool any = false;
    for (int& v : h->variantOf) { v = remap[v]; any = any || v != 0; }
    if (!any) h->variantOf.clear();
    return 0;
}

int avdsp_b200_coef_words(const int32_t* prog, int progWords, int format, int32_t* wordIndex, int maxOut) {
    return tableWords(&Lowered::coefWords, false, prog, progWords, format, wordIndex, maxOut);
}

int avdsp_b200_set_coefs(avdsp_b200_t* h, int firstStream, int nStreams, const int32_t* values, int memspace, void* cudaStream) {
    const char* overlap = h && !h->L.coefTableOk ? "biquad parameter blocks of this program overlap: no coefficient table" : nullptr;
    return setRows(h, &avdsp_b200::coefTab, overlap, firstStream, nStreams, values, memspace, cudaStream);
}

// validated at every rate the program admits, as the header states (avdsp_b200_coef_words: at the lowest one)
int avdsp_b200_fir_tap_words(const int32_t* prog, int progWords, int format, int32_t* wordIndex, int maxOut) {
    return tableWords(&Lowered::firTapWords, true, prog, progWords, format, wordIndex, maxOut);
}

int avdsp_b200_set_fir_taps(avdsp_b200_t* h, int firstStream, int nStreams, const int32_t* values, int memspace, void* cudaStream) {
    return setRows(h, &avdsp_b200::firTab, nullptr, firstStream, nStreams, values, memspace, cudaStream);
}

int avdsp_b200_num_variants(const avdsp_b200_t* h) {
    if (!h) return 0;
    int n = h->shards.empty() ? 1 + (int)h->variants.size() : 0;
    for (const avdsp_b200* sh : h->shards) n += 1 + (int)sh->variants.size();
    return n;
}

int avdsp_b200_reload_params(avdsp_b200_t* h, const int32_t* prog, int progWords) {
    if (!h || !prog) return setErr(AVDSP_B200_ERR_ARG, "NULL argument");
    std::string err;
    const int rc = relowerProgram(prog, progWords, &h->L, &err);
    if (rc < 0) return setErr(rc, err);
    if (!h->shards.empty()) {
        const int r = forShards(h, [&](int, avdsp_b200* sh) { return std::min(0, avdsp_b200_reload_params(sh, prog, progWords)); });
        return r < 0 ? r : rc;
    }
    { const int q = quiesce(h); if (q < 0) return q; }
    h->variants.clear();                                      // a new program for everybody: per-stream overrides start over
    h->variantOf.clear();
    freeTable(h->coefTab);                                    // ... the tables too
    freeTable(h->firTab);
    if (h->dFirFlags) { cudaFree(h->dFirFlags); h->dFirFlags = nullptr; }
    if (h->dFirTcPer) { cudaFree(h->dFirTcPer); h->dFirTcPer = nullptr; }
    h->firTcPerValid = h->firTcPerFailed = false;
    const int r = uploadPlanData(*h, h->device, h->nStreams, h->numSMs);
    return r < 0 ? r : rc;
}

int avdsp_b200_get_state(avdsp_b200_t* h, int stream, int32_t* words) {
    if (!h || !words || stream < 0 || stream >= h->nStreams) return setErr(AVDSP_B200_ERR_ARG, "bad stream index");
    if (!h->shards.empty()) { const int k = shardOf(h, stream); return avdsp_b200_get_state(h->shards[k], stream - h->shardFirst[k], words); }
    { const int q = quiesce(h); if (q < 0) return q; }
    const int W = h->L.gen.h.stateWords;
    CU(cudaMemcpy(words, h->dState + (size_t)stream * W, (size_t)W * 4, cudaMemcpyDeviceToHost));
    return 0;
}
int avdsp_b200_set_state(avdsp_b200_t* h, int stream, const int32_t* words) {
    if (!h || !words || stream < 0 || stream >= h->nStreams) return setErr(AVDSP_B200_ERR_ARG, "bad stream index");
    if (!h->shards.empty()) { const int k = shardOf(h, stream); return avdsp_b200_set_state(h->shards[k], stream - h->shardFirst[k], words); }
    { const int q = quiesce(h); if (q < 0) return q; }
    const int W = h->L.gen.h.stateWords;
    CU(cudaMemcpy(h->dState + (size_t)stream * W, words, (size_t)W * 4, cudaMemcpyHostToDevice));
    return 0;
}

double avdsp_b200_measure_int_peak(int device, int iters) {
    if (cudaSetDevice(device) != cudaSuccess) { setErr(AVDSP_B200_ERR_CUDA, "no CUDA device"); return 0.0; }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return 0.0;
    long long* d = nullptr;
    if (cudaMalloc(&d, 8) != cudaSuccess) return 0.0;
    const int blocks = prop.multiProcessorCount * 8, threads = 256;
    cudaEvent_t a, b; cudaEventCreate(&a); cudaEventCreate(&b);
    k_int_peak<<<blocks, threads>>>(d, iters / 8 + 1, 3, 5);          // warm-up
    double best = 0.0;
    for (int rep = 0; rep < 3; rep++) {
        cudaEventRecord(a);
        k_int_peak<<<blocks, threads>>>(d, iters, 3 + rep, 5);
        cudaEventRecord(b);
        if (cudaEventSynchronize(b) != cudaSuccess) { best = 0.0; break; }
        float ms = 0; cudaEventElapsedTime(&ms, a, b);
        const double rate = (double)blocks * threads * 8.0 * iters / (ms * 1e-3);
        best = std::max(best, rate);
    }
    cudaEventDestroy(a); cudaEventDestroy(b); cudaFree(d);
    return best;
}

double avdsp_b200_measure_f32_peak(int device, int iters, int packed) {
    if (cudaSetDevice(device) != cudaSuccess) { setErr(AVDSP_B200_ERR_CUDA, "no CUDA device"); return 0.0; }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return 0.0;
    float* d = nullptr;
    if (cudaMalloc(&d, 8) != cudaSuccess) return 0.0;
    const int blocks = prop.multiProcessorCount * 8, threads = 256;
    cudaEvent_t a, b; cudaEventCreate(&a); cudaEventCreate(&b);
    double best = 0.0;
    for (int rep = 0; rep < 4; rep++) {
        cudaEventRecord(a);
        if (packed) k_f32_peak<1><<<blocks, threads>>>(d, iters, -0.0003f); else k_f32_peak<0><<<blocks, threads>>>(d, iters, -0.0003f);
        cudaEventRecord(b);
        if (cudaEventSynchronize(b) != cudaSuccess) { best = 0.0; break; }
        float ms = 0; cudaEventElapsedTime(&ms, a, b);
        const double rate = (double)blocks * threads * 8.0 * (packed ? 2.0 : 1.0) * iters / (ms * 1e-3);
        if (rep) best = std::max(best, rate);
    }
    cudaEventDestroy(a); cudaEventDestroy(b); cudaFree(d);
    return best;
}

} // extern "C"

// =============================================================================================
// Reference entry points (per-frame compatibility path).  One live program per process, exactly
// like the reference (dspHeaderPtr and the fs/TPDF globals are file-scope there).
// =============================================================================================
namespace {
struct Compat {
    int32_t* code = nullptr;
    int maxSize = 0, total = 0, dataSize = 0;
    int fs = 0, seed = 0, dither = 0, format = 0;
    bool haveReset = false;
    avdsp_b200* h = nullptr;
    GenericPlan plan;                 // the program's plan with an identity 32-slot io map
    int* dIo = nullptr;               // 32 in + 32 out words on the device
    std::vector<int32_t> stateHost;
} g_compat;

int compatFormatGuess(const int32_t* code) { return ((uint32_t)code[H_FORMAT] & 0xFFFF) ? FMT_INT64 : FMT_FLOAT; }

int compatBuild(int format) {
    Compat& C = g_compat;
    if (C.h) { avdsp_b200_destroy(C.h); C.h = nullptr; }
    if (C.dIo) { cudaFree(C.dIo); C.dIo = nullptr; }
    const int32_t seed = C.seed;
    const int rc = avdsp_b200_create(&C.h, C.code, C.total, C.fs, format, 1, &seed, C.dither, 0);
    if (rc < 0) return rc;
    C.format = format;
    C.plan = C.h->L.gen;
    C.plan.h.nIn = C.plan.h.nOut = kIoSlots;
    for (int k = 0; k < kIoSlots; k++) C.plan.h.inIdx[k] = C.plan.h.outIdx[k] = (uint8_t)k;
    CU(cudaMalloc(&C.dIo, 2 * kIoSlots * 4));
    C.stateHost.assign(C.plan.h.stateWords, 0);
    return rc;
}

int compatRun(int format, int32_t* corePtr, int* rundata, void* io) {
    Compat& C = g_compat;
    if (!C.code || !C.haveReset) return setErr(AVDSP_B200_ERR_ARG, "dspRuntime called before dspRuntimeInit/dspRuntimeReset");
    if (!C.h || C.format != format) { const int rc = compatBuild(format); if (rc < 0) return rc; }
    avdsp_b200* h = C.h;
    // live parameter patching: the reference re-reads the program every frame
    if (memcmp(C.code, h->L.words.data(), (size_t)C.total * 4) != 0) {
        const int rc = avdsp_b200_reload_params(h, C.code, C.total);
        if (rc < 0) return rc;
        const GenericPlan keep = C.plan;
        C.plan = h->L.gen;
        C.plan.h.nIn = keep.h.nIn; C.plan.h.nOut = keep.h.nOut;
        memcpy(C.plan.h.inIdx, keep.h.inIdx, sizeof keep.h.inIdx); memcpy(C.plan.h.outIdx, keep.h.outIdx, sizeof keep.h.outIdx);
    }
    const long word = corePtr - C.code;
    int core = -1;
    for (size_t c = 0; c < h->L.cores.size(); c++)
        if (h->L.cores[c].coreWord == word || h->L.cores[c].beginWord == word) { core = (int)c; break; }
    if (core < 0) return setErr(AVDSP_B200_ERR_ARG, "core pointer does not designate a DSP_CORE of the loaded program");
    const PlanHeader& P = C.plan.h;
    CU(cudaSetDevice(h->device));
    // the caller owns the data area and the MEM words: device copy follows the caller's buffer
    if (rundata && P.dataSize) CU(cudaMemcpyAsync(h->dState, rundata, (size_t)P.dataSize * 4, cudaMemcpyHostToDevice, h->stream));
    if (P.nMem) {
        for (int k = 0; k < P.nMem; k++) { C.stateHost[2 * k] = C.code[h->L.memWord[k]]; C.stateHost[2 * k + 1] = C.code[h->L.memWord[k] + 1]; }
        CU(cudaMemcpyAsync(h->dState + P.memOff, C.stateHost.data(), (size_t)P.nMem * 8, cudaMemcpyHostToDevice, h->stream));
    }
    CU(cudaMemcpyAsync(C.dIo, io, kIoSlots * 4, cudaMemcpyHostToDevice, h->stream));
    const int r = launchRange(h, C.dIo, C.dIo + kIoSlots, 1, AVDSP_B200_INTERLEAVED, 0, 1, h->stream, core, &C.plan);
    if (r < 0) return r;
    CU(cudaMemcpyAsync(io, C.dIo + kIoSlots, kIoSlots * 4, cudaMemcpyDeviceToHost, h->stream));
    if (rundata && P.dataSize) CU(cudaMemcpyAsync(rundata, h->dState, (size_t)P.dataSize * 4, cudaMemcpyDeviceToHost, h->stream));
    if (P.nMem) CU(cudaMemcpyAsync(C.stateHost.data(), h->dState + P.memOff, (size_t)P.nMem * 8, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    for (int k = 0; k < P.nMem; k++) {       // STORE_MEM lands in the caller's code area (runtime/dsp_runtime.c:760-766)
        const int w = h->L.memWord[k];
        C.code[w] = C.stateHost[2 * k]; C.code[w + 1] = C.stateHost[2 * k + 1];
        h->L.words[w] = C.code[w]; h->L.words[w + 1] = C.code[w + 1];
    }
    return 0;
}
} // namespace

extern "C" {

int dspRuntimeReset(const int fs, int random, int defaultDither) {
    Compat& C = g_compat;
    if (!C.code) return setErr(-1, "dspRuntimeReset before dspRuntimeInit");
    const int fi = freqToIndex(fs);
    if (fi >= kNumFreq) return setErr(-1, "sampling frequency not supported");
    if (fi < C.code[H_FREQMIN] || fi > C.code[H_FREQMAX]) return setErr(-2, "sampling freq not compatible with encoded dsp program");
    C.fs = fs; C.seed = random; C.dither = defaultDither; C.haveReset = true;
    // the reference clears the data area that follows the code (runtime/dsp_runtime.c:137-141)
    memset(C.code + C.total, 0, (size_t)C.dataSize * 4);
    if (C.h) { avdsp_b200_destroy(C.h); C.h = nullptr; }       // rebuilt lazily for the format of the first dspRuntime_<fmt> call
    return 0;
}

int dspRuntimeInit(int32_t* codePtr, int maxSize, const int fs, int random, int defaultDither) {
    Compat& C = g_compat;
    if (!codePtr || wordOpcode(codePtr[0]) != OP_HEADER) return setErr(-1, "no dsp header in this program");
    const int total = codePtr[H_TOTAL], dsz = codePtr[H_DATASIZE];
    if (total < H_WORDS || dsz < 0 || (long long)total + dsz > (long long)maxSize) return setErr(-6, "program+data is over the allowed size");
    // validation only (no device work yet): lower for the first frequency the program covers
    Lowered tmp; std::string err;
    const int fmin = codePtr[H_FREQMIN];
    const int vfs = (fmin >= 0 && fmin < kNumFreq) ? kFreqTable[fmin] : 0;
    const int rc = decodeProgram(codePtr, total, maxSize, compatFormatGuess(codePtr), vfs, defaultDither, &tmp, &err);
    if (rc < 0) return setErr(rc, err);
    if (C.h) { avdsp_b200_destroy(C.h); C.h = nullptr; }
    C.code = codePtr; C.maxSize = maxSize; C.total = total; C.dataSize = dsz; C.haveReset = false;
    if (fs) { const int r = dspRuntimeReset(fs, random, defaultDither); if (r) return r; }
    return total;
}

int32_t* dspFindCore(int32_t* codePtr, const int numCore) {
    if (!codePtr) return nullptr;
    const int w = findCoreWord(codePtr, numCore);
    return w < 0 ? nullptr : codePtr + w;
}
int32_t* dspFindCoreBegin(int32_t* corePtr) {
    if (!corePtr) return nullptr;
    return corePtr + findCoreBeginWord(corePtr, 0);
}

int dspRuntime_2(int32_t* c, int* d, void* io) { return compatRun(FMT_INT64, c, d, io); }
int dspRuntime_3(int32_t* c, int* d, void* io) { return compatRun(FMT_FLOAT, c, d, io); }
int dspRuntime_4(int32_t* c, int* d, void* io) { return compatRun(FMT_DOUBLE, c, d, io); }
int dspRuntime_5(int32_t* c, int* d, void* io) { return compatRun(FMT_FLOAT_FLOAT, c, d, io); }
int dspRuntime_6(int32_t* c, int* d, void* io) { return compatRun(FMT_DOUBLE_FLOAT, c, d, io); }

// DSP_QNM family (runtime/dsp_header.h:276-285): x -> fixed point with m mantissa bits in a b-bit
// container, saturating at the container limits, truncating toward zero.
static long long qmb(double x, int m, int b) {
    if (m >= b || b > 64 || m < 1) return 0;                       // the macro divides by zero here
    const double lim = (double)(1ULL << (b - m - 1));
    if (x >= lim) return b >= 64 ? 9223372036854775807LL : (long long)((1ULL << (b - 1)) - 1);
    if (-x > lim) return b >= 64 ? (-9223372036854775807LL - 1LL) : (long long)(1ULL << (b - 1));   // positive magnitude, as the macro yields
    if (b >= 33) return (long long)(x * (double)(1LL << m));
    return (long long)(int)(x * (double)(1L << m));
}
long long dspQNM(double x, int n, int m) { return qmb(x, m, n + m); }
long long dspQM64(double x, int m) { return qmb(x, m, 64); }
int dspQM32(double x, int m) { return (int)qmb(x, m, 32); }

const char* dspOpcodeText[AVDSP_B200_MAX_OPCODE] = {
    "DSP_END_OF_CODE", "\nDSP_HEADER", "DSP_NOP", "\nDSP_CORE", "\nDSP_PARAM", "\nDSP_PARAM_NUM", "DSP_SERIAL",
    "DSP_TPDF_CALC", "DSP_TPDF", "DSP_WHITE", "DSP_CLRXY", "DSP_SWAPXY", "DSP_COPYXY", "DSP_COPYYX",
    "DSP_ADDXY", "DSP_ADDYX", "DSP_SUBXY", "DSP_SUBYX", "DSP_MULXY", "DSP_DIVXY", "DSP_DIVYX", "DSP_AVGXY", "DSP_AVGYX",
    "DSP_NEGX", "DSP_NEGY", "DSP_SQRTX", "DSP_SHIFT", "DSP_VALUE", "DSP_VALUE_INT", "DSP_MUL_VALUE", "DSP_MUL_VALUE_INT",
    "DSP_DIV_VALUE", "DSP_DIV_VALUE_INT", "DSP_AND_VALUE_INT",
    "DSP_LOAD", "DSP_LOAD_GAIN", "DSP_LOAD_MUX", "DSP_STORE", "DSP_LOAD_STORE", "DSP_LOAD_MEM", "DSP_STORE_MEM",
    "DSP_GAIN", "DSP_SAT0DB", "DSP_SAT0DB_TPDF", "DSP_SAT0DB_GAIN", "DSP_SAT0DB_TPDF_GAIN",
    "DSP_DELAY_1", "DSP_DELAY", "DSP_DELAY_DP", "DSP_DATA_TABLE", "DSP_BIQUADS", "DSP_FIR",
    "DSP_RMS", "DSP_DCBLOCK", "DSP_DITHER", "DSP_DITHER_NS2", "DSP_DISTRIB", "DSP_DIRAC", "DSP_SQUAREWAVE", "DSP_CLIP",
    "DSP_LOAD_MEM_DATA", "DSP_SINE",
};

} // extern "C"

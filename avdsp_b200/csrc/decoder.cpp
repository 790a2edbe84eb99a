// decoder.cpp -- validate + lower an AVDSP program.  See decoder.h / plan.h.
//
// Reference behaviour being restated (citations: /root/reference/module_avdsp/):
//   validation      runtime/dsp_runtime.c:150-195 (dspRuntimeInit), :116-145 (dspRuntimeReset),
//                   runtime/dsp_header.h:234-251 (dspCalcSumCore)
//   core discovery  runtime/dsp_runtime.c:42-77  (dspFindCore, dspFindCoreBegin)
//   operand decode  runtime/dsp_runtime.c:302-1314, one `case` per opcode
//   PARAM layouts   encoder/dsp_encoder.c (biquads :1225-1290, mux :798-813, delay :1088-1160)
#include "decoder.h"
#include <cstdio>
#include <cstring>
#include <algorithm>
#include <map>
#include <memory>

namespace avdsp {

namespace {

struct Fail { int code; std::string msg; };

struct Ctx {
    Lowered* L;
    const int32_t* w;       // program words
    int total;
    uint32_t delayFactor;
    int nMemSlots = 0;
    std::map<int, int> memSlotOfWord;
    std::vector<std::pair<int, int>> biquadBlocks;      // (parameter block word, sections) of every DSP_BIQUADS, bypassed too
    std::vector<std::pair<int, int>> firBlocks;         // (first tap word, taps) of every DSP_FIR convolution entry, every fs column
    std::vector<std::pair<int, int>> firConvs;          // (micro-op index, first tap word) of every lowered FIR convolution

    [[noreturn]] void fail(int code, const char* fmt, int a = 0, int b = 0) {
        char buf[256]; snprintf(buf, sizeof buf, fmt, a, b);
        throw Fail{code, buf};
    }
    int32_t code(int idx, int atOp) {
        if (idx < 0 || idx >= total) fail(ERR_MALFORMED, "opcode at word %d points outside the program (%d)", atOp, idx);
        return w[idx];
    }
    void checkData(int off, int64_t n, int atOp) {      // 64-bit: off + n must not wrap for offsets near INT_MAX
        if (off < 0 || n < 0 || (int64_t)off + n > (int64_t)L->dataSize) fail(ERR_MALFORMED, "opcode at word %d: data offset %d outside the data area", atOp, off);
    }
    void checkIo(int io, int atOp) {
        if (io < 0 || io >= kIoSlots) fail(ERR_MALFORMED, "opcode at word %d: io index %d out of range", atOp, io);
    }
    int pool(int32_t v) {
        GenericPlan& g = L->gen;
        if (g.h.nPool >= kMaxPool) fail(ERR_PLAN_SIZE, "plan pool full (%d words)", kMaxPool);
        g.pool[g.h.nPool] = v;
        return g.h.nPool++;
    }
    void emit(int op, int n, int32_t a, int32_t b, int32_t c) {
        GenericPlan& g = L->gen;
        if (g.h.nOps >= kMaxOps) fail(ERR_PLAN_SIZE, "plan has more than %d micro-ops", kMaxOps);
        MicroOp& m = g.ops[g.h.nOps++];
        m.op = (uint16_t)op; m.n = (uint16_t)n; m.a = a; m.b = b; m.c = c;
    }
    int memSlot(int wordIdx, int atOp) {
        if (wordIdx < 0 || wordIdx + 1 >= total) fail(ERR_MALFORMED, "opcode at word %d: MEM location %d outside the program", atOp, wordIdx);
        auto it = memSlotOfWord.find(wordIdx);
        if (it != memSlotOfWord.end()) return it->second;
        int s = nMemSlots++;
        memSlotOfWord[wordIdx] = s;
        L->memWord.push_back(wordIdx);
        return s;
    }
};

int aluWords(int aluClass) { return aluClass == ALU_F32 ? 1 : 2; }

// Lower the opcodes of one core: [begin, next DSP_CORE / END_OF_CODE)
void lowerCore(Ctx& cx, int begin) {
    Lowered* L = cx.L;
    const int32_t* w = cx.w;
    const int aw = aluWords(L->gen.h.aluClass);
    int p = begin;
    for (;;) {
        if (p < 0 || p >= cx.total) cx.fail(ERR_MALFORMED, "opcode walk left the program at word %d", p);
        const int op = wordOpcode(w[p]), skip = wordSkip(w[p]);
        if (skip == 0 || op == OP_CORE) return;            // dsp_runtime.c:321-331
        if (p + skip > cx.total) cx.fail(ERR_MALFORMED, "opcode at word %d overruns the program", p);
        auto arg = [&](int k) -> int32_t {
            if (k + 1 >= skip && !(op == OP_DELAY || op == OP_DELAY_DP)) cx.fail(ERR_MALFORMED, "opcode at word %d: missing argument %d", p, k);
            return cx.code(p + 1 + k, p);
        };
        switch (op) {
        case OP_HEADER: case OP_NOP: case OP_PARAM: case OP_PARAM_NUM: case OP_SERIAL:
            break;                                          // skipped at run time (:333,852-868)
        case OP_SWAPXY: case OP_COPYXY: case OP_COPYYX: case OP_CLRXY:
        case OP_ADDXY: case OP_ADDYX: case OP_SUBXY: case OP_SUBYX: case OP_MULXY:
        case OP_DIVXY: case OP_DIVYX: case OP_AVGXY: case OP_AVGYX: case OP_NEGX: case OP_NEGY:
        case OP_SQRTX: case OP_SAT0DB: case OP_SAT0DB_TPDF: case OP_WHITE:
            cx.emit(op, 0, 0, 0, 0); break;
        case OP_SHIFT: case OP_MUL_VALUE: case OP_MUL_VALUE_INT: case OP_DIV_VALUE:
        case OP_DIV_VALUE_INT: case OP_AND_VALUE_INT: case OP_CLIP:
            cx.emit(op, 0, arg(0), 0, 0); break;            // immediate below the opcode
        case OP_GAIN: case OP_SAT0DB_GAIN: case OP_SAT0DB_TPDF_GAIN: case OP_VALUE: case OP_VALUE_INT:
            cx.emit(op, 0, cx.code(p + arg(0), p), 0, 0); break;   // relative pointer -> immediate
        case OP_TPDF_CALC: case OP_TPDF: {
            int d = arg(0); if (d == 0) d = L->defaultDither;      // dsp_tpdf.h:56
            cx.checkData(arg(1), aw, p);
            cx.emit(op, 0, d, arg(1), 0); break; }
        case OP_LOAD: case OP_STORE:
            cx.checkIo(arg(0), p); cx.emit(op, 0, arg(0), 0, 0); break;
        case OP_LOAD_GAIN:
            cx.checkIo(arg(0), p); cx.emit(op, 0, arg(0), cx.code(p + arg(1), p), 0); break;
        case OP_LOAD_MUX: {
            int t = p + arg(0);
            int n = (int16_t)(cx.code(t, p) & 0xFFFF);
            if (n < 0) n = 0;
            int first = L->gen.h.nPool;
            for (int k = 0; k < n; k++) {
                int io = cx.code(t + 1 + 2 * k, p); cx.checkIo(io, p);
                cx.pool(io); cx.pool(cx.code(t + 2 + 2 * k, p));
            }
            cx.checkData(arg(1), aw, p);
            cx.emit(op, n, first, arg(1), 0); break; }
        case OP_LOAD_STORE: {
            int n = (skip - 1) / 2, first = L->gen.h.nPool;
            for (int k = 0; k < n; k++) {
                int i = arg(2 * k), o = arg(2 * k + 1); cx.checkIo(i, p); cx.checkIo(o, p);
                cx.pool(i); cx.pool(o);
            }
            cx.emit(op, n, first, 0, 0); break; }
        case OP_LOAD_MEM: case OP_STORE_MEM:
            cx.emit(op, 0, cx.memSlot(p + arg(0), p), 0, 0); break;   // slot index, turned into an offset later
        case OP_LOAD_MEM_DATA:
            cx.checkData(arg(0), aw, p); cx.emit(op, 0, arg(0), 0, 0); break;
        case OP_DELAY_1:
            cx.checkData(arg(0), aw, p); cx.emit(op, 0, arg(0), 0, 0); break;
        case OP_DELAY: case OP_DELAY_DP: {                  // :769-824
            uint32_t maxSize = (uint32_t)arg(0);
            int off = arg(1), rel = arg(2);
            uint32_t n;
            if (rel == 0) n = (uint32_t)(((uint64_t)maxSize * cx.delayFactor) >> 32);
            else {
                uint32_t us = (uint32_t)cx.code(p + rel, p) & 0xFFFFu;
                n = (uint32_t)(((uint64_t)us * cx.delayFactor) >> 32);
                if (n > maxSize) n = maxSize;
            }
            if (n == 0) break;                              // "sanity check ... delay=0 to bypass it"
            cx.checkData(off, 1 + (int64_t)n * (op == OP_DELAY_DP ? aw : 1), p);
            cx.emit(op, 0, off, (int32_t)n, 0); break; }
        case OP_BIQUADS: {                                  // :827-849
            int off = arg(0), h = p + arg(1);
            int num = (int16_t)(cx.code(h, p) & 0xFFFF);
            if (num > 0) cx.biquadBlocks.emplace_back(h, num);
            if (cx.code(h + 1, p) == 0 || num <= 0) break;  // bypass flag: X untouched
            cx.checkData(off, 6 * num, p);
            int stride = 2 + 6 * L->nFreq, c0 = h + 5 + 6 * L->fsRel;
            int first = L->gen.h.nPool;
            for (int s = 0; s < num; s++)
                for (int k = 0; k < 5; k++) cx.pool(cx.code(c0 + s * stride + k, p));
            cx.emit(op, num, off, first, h); break; }     // c: the block's word until lowerAll makes it a table column
        case OP_FIR: {                                      // :928-969
            // the tap blocks of every fs column are columns of the per-stream FIR table; only this rate's entry is lowered
            for (int f = 0; f < L->nFreq && f + 1 < skip; f++) {
                const int32_t r = w[p + 1 + f];
                const int64_t t = (int64_t)p + r;
                if (r == 0 || t < 0 || t >= cx.total) continue;
                if (w[t] > 0 && (w[t] >> 16) == 0) cx.firBlocks.emplace_back((int)t + 1, w[t]);
            }
            int rel = arg(L->fsRel);
            if (rel == 0) break;
            int off = arg(L->nFreq);
            int t = p + rel;
            int lw = cx.code(t, p), delay = lw >> 16;
            if (delay) {
                if (delay < 0) cx.fail(ERR_MALFORMED, "opcode at word %d: negative FIR delay", p);
                cx.checkData(off, 1 + (int64_t)delay, p);
                cx.emit(OP_FIR, 0, off, delay, 0);          // n==0: plain ring delay of `delay` samples
            } else if (lw > 0) {
                cx.checkData(off, lw, p);
                cx.code(t + lw, p);                          // bounds
                FirDesc fd; fd.tapsOff = (int)L->bigPool.size(); fd.length = lw; fd.stateOff = off;
                for (int k = 0; k < lw; k++) L->bigPool.push_back(w[t + 1 + k]);
                L->firs.push_back(fd);
                cx.firConvs.emplace_back(L->gen.h.nOps, t + 1);
                cx.emit(OP_FIR, 1, off, fd.tapsOff, lw);    // n==1: convolution, b=taps offset, c=length
            }
            break; }
        case OP_DATA_TABLE: {                               // :900-923
            int div = arg(1), size = arg(2), idxOff = arg(3), t = p + arg(4);
            if (size <= 0 || size > cx.total) cx.fail(ERR_MALFORMED, "opcode at word %d: data table size %d", p, size);
            // index += div; if (index >= size) index -= size (:911-912) only stays inside the table for 0 <= div < size
            if (div < 0 || div >= size) cx.fail(ERR_MALFORMED, "opcode at word %d: data table divider %d outside [0, size)", p, div);
            cx.code(t, p); cx.code(t + size - 1, p);
            cx.checkData(idxOff, 1, p);
            int first = L->gen.h.nPool;
            cx.pool(arg(0)); cx.pool(arg(1)); cx.pool(size); cx.pool(idxOff); cx.pool((int)L->bigPool.size());
            for (int k = 0; k < size; k++) L->bigPool.push_back(w[t + k]);
            cx.emit(op, 0, first, 0, 0); break; }
        case OP_DCBLOCK:
            cx.checkData(arg(0), aw + 2, p); cx.emit(op, 0, arg(0), arg(1 + L->fsRel), 0); break;
        case OP_DITHER:
            cx.checkData(arg(0), 3 * aw, p); cx.emit(op, 0, arg(0), 0, 0); break;
        case OP_DITHER_NS2: {
            cx.checkData(arg(0), 3, p);
            int t = p + arg(1) + 3 * L->fsRel, first = L->gen.h.nPool;
            for (int k = 0; k < 3; k++) cx.pool(cx.code(t + k, p));
            cx.emit(op, 0, arg(0), first, 0); break; }
        case OP_RMS: {
            int off = arg(0), delay = arg(1);
            if (delay < 0) cx.fail(ERR_MALFORMED, "opcode at word %d: negative RMS delay", p);
            cx.checkData(off, 5 + 2 * (int64_t)aw + (int64_t)delay * aw, p);
            int first = L->gen.h.nPool;
            cx.pool(arg(2 + 2 * L->fsRel)); cx.pool(arg(3 + 2 * L->fsRel));
            cx.emit(op, 0, off, delay, first); break; }
        case OP_DISTRIB:
            cx.checkIo(arg(0), p);
            if (arg(1) < 2) cx.fail(ERR_MALFORMED, "opcode at word %d: DISTRIB size < 2", p);
            cx.checkData(arg(2), 1 + (int64_t)arg(1), p);
            cx.emit(op, 0, arg(0), arg(1), arg(2)); break;
        case OP_DIRAC: case OP_SQUAREWAVE:
            cx.checkData(arg(0), 1, p); cx.emit(op, 0, arg(0), arg(1), arg(2 + L->fsRel)); break;
        case OP_SINE:   // WIP in the reference: the case does not compile at HEAD (SURVEY.md App. C #1) and is
            break;      // an empty `break` in the buildable reference the oracle pins (oracle/Makefile patch b): no-op
        default:
            cx.fail(ERR_OPCODE_NEW, "unknown opcode %d at word %d", op, p);
        }
        p += skip;
    }
}

// ---- chain recognition ------------------------------------------------------------------------
struct ChainFail { std::string why; };

int chainPool(ChainPlan& c, int32_t v) {
    if (c.h.nPool >= kMaxChainPool) throw ChainFail{"chain pool full"};
    c.pool[c.h.nPool] = v; return c.h.nPool++;
}

void buildChainPlan(Lowered* L) {
    const GenericPlan& g = L->gen;
    ChainPlan& c = L->chain;
    memset(&c, 0, sizeof c);
    c.h.format = g.h.format; c.h.aluClass = g.h.aluClass; c.h.sampleInt = g.h.sampleInt;
    c.h.nIn = g.h.nIn; c.h.nOut = g.h.nOut;
    c.h.dataSize = g.h.dataSize; c.h.stateWords = g.h.stateWords; c.h.auxOff = g.h.auxOff;
    c.h.storeDither = g.h.defaultDither;
    for (int k = 0; k < kIoSlots; k++) c.h.chainOfOut[k] = -1;
    if (!g.h.sampleInt && g.h.aluClass != ALU_F32) throw ChainFail{"DSP_FORMAT 6 (float samples, double ALU) runs on the generic executor"};

    int inChOfSlot[kIoSlots], outChOfSlot[kIoSlots];
    for (int k = 0; k < kIoSlots; k++) inChOfSlot[k] = outChOfSlot[k] = -1;
    for (int k = 0; k < g.h.nIn; k++)  inChOfSlot[g.h.inIdx[k]] = k;
    for (int k = 0; k < g.h.nOut; k++) outChOfSlot[g.h.outIdx[k]] = k;
    // every io slot written anywhere in the program
    uint32_t written = 0;
    for (int i = 0; i < g.h.nOps; i++) {
        const MicroOp& m = g.ops[i];
        if (m.op == OP_STORE || m.op == OP_DISTRIB) written |= 1u << m.a;
        if (m.op == OP_LOAD_STORE) for (int k = 0; k < m.n; k++) written |= 1u << g.pool[m.a + 2 * k + 1];
    }
    auto inputCh = [&](int slot) -> int {
        if ((written >> slot) & 1u) throw ChainFail{"an input slot is also written by the program (io hand-off between paths)"};
        if (inChOfSlot[slot] < 0) return -1;    // never fed by the host: reads 0
        return inChOfSlot[slot];
    };

    // the path being built (chain index nChains) stores to output channel ch; a later path of the frame that stores to the
    // same slot wins: the earlier STORE is dead (its path still runs for its state)
    auto claimOutput = [&](int ch, ChainDesc& d) {
        const int owner = c.h.chainOfOut[ch];
        if (owner == c.h.nChains) return;
        if (owner >= 0) {
            ChainDesc& o = c.chains[owner];
            int w = 0;
            for (int k = 0; k < o.nStores; k++) if (o.storeCh[k] != ch) o.storeCh[w++] = o.storeCh[k];
            o.nStores = (uint8_t)w;
        }
        c.h.chainOfOut[ch] = c.h.nChains;
        d.storeCh[d.nStores++] = (uint8_t)ch;
    };
    struct MemProducer { int srcKind, srcCh, srcArg, consumers; std::vector<int> secOff; std::vector<int32_t> coefs; std::vector<int> cols; };
    std::vector<std::pair<int, MemProducer>> producers;          // keyed by the MEM word's state offset
    auto findProducer = [&](int memOff) -> MemProducer* { for (auto& pr : producers) if (pr.first == memOff) return &pr.second; return nullptr; };
    for (int core = 0; core < g.h.nCores; core++) {
        int i = g.h.coreStart[core], e = g.h.coreStart[core + 1];
        auto takeRaw = [&]() {
            // DSP_LOAD_STORE (dsp_runtime.c:738-747): raw io[out] = io[in] copies; each pair is a pass-through path
            const MicroOp& s = g.ops[i];
            for (int k = 0; k < s.n; k++) {
                if (c.h.nChains >= kMaxChains) throw ChainFail{"more than kMaxChains signal paths"};
                ChainDesc& d = c.chains[c.h.nChains];
                memset(&d, 0, sizeof d);
                d.muxStateOff = -1; d.delayOff = -1; d.srcId = -1; d.accRow = -1;
                d.srcKind = SRC_RAW; d.srcCh = (int16_t)inputCh(g.pool[s.a + 2 * k]);
                const int ch = outChOfSlot[g.pool[s.a + 2 * k + 1]];
                if (ch < 0) throw ChainFail{"LOAD_STORE to a slot outside the declared outputs"};
                claimOutput(ch, d);
                c.h.nChains++; c.h.nRaw++;
            }
            i++;
        };
        // core 1 may compute the frame's dither after raw copies (the DAC8PRO firmware does): LOAD_STORE neither uses the
        // TPDF value nor the STORE mask, so TPDF_CALC behind them is still "at the start of the frame" for everything else
        while (core == 0 && i < e && g.ops[i].op == OP_LOAD_STORE && c.h.nChains == c.h.nRaw && !c.h.hasTpdfCalc) takeRaw();
        if (i < e && g.ops[i].op == OP_TPDF_CALC) {
            if (core != 0 || c.h.nChains != c.h.nRaw || c.h.hasTpdfCalc) throw ChainFail{"TPDF_CALC not at the very start of core 1"};
            c.h.hasTpdfCalc = 1; c.h.tpdfDither = g.ops[i].a; c.h.tpdfDataOff = g.ops[i].b;
            c.h.storeDither = g.ops[i].a;
            i++;
        }
        while (i < e) {
            if (g.ops[i].op == OP_LOAD_STORE) { takeRaw(); continue; }
            if (c.h.nChains >= kMaxChains) throw ChainFail{"more than kMaxChains signal paths"};
            ChainDesc& d = c.chains[c.h.nChains];
            memset(&d, 0, sizeof d);
            d.muxStateOff = -1; d.delayOff = -1;
            const MicroOp& s = g.ops[i];
            if (s.op == OP_LOAD)           { d.srcKind = SRC_LOAD;      d.srcCh = (int16_t)inputCh(s.a); }
            else if (s.op == OP_LOAD_GAIN) { d.srcKind = SRC_LOAD_GAIN; d.srcCh = (int16_t)inputCh(s.a); d.srcArg = s.b; }
            else if (s.op == OP_LOAD_MUX) {
                d.srcKind = SRC_LOAD_MUX; d.srcCh = (int16_t)s.n; d.muxStateOff = s.b;
                d.srcArg = c.h.nPool;
                for (int k = 0; k < s.n; k++) { chainPool(c, inputCh(g.pool[s.a + 2 * k])); chainPool(c, g.pool[s.a + 2 * k + 1]); }
            }
            std::vector<int> secOff, cols;
            std::vector<int32_t> coefs;
            if (s.op == OP_LOAD_MEM) {
                // a cascade continued from an earlier core through a MEM word: inline the producer (same frame, canonical order:
                // the consumer's BIQUADS sees x = MEM >> 28 = the producer's last y, exactly as if the sections were consecutive)
                MemProducer* pr = findProducer(s.a);
                if (!pr) throw ChainFail{"LOAD_MEM of a word no earlier cascade of the frame stored"};
                d.srcKind = (uint8_t)pr->srcKind; d.srcCh = (int16_t)pr->srcCh; d.srcArg = pr->srcArg;
                secOff = pr->secOff; coefs = pr->coefs; cols = pr->cols; pr->consumers++;
            } else if (s.op != OP_LOAD && s.op != OP_LOAD_GAIN && s.op != OP_LOAD_MUX)
                throw ChainFail{"a signal path does not start with LOAD / LOAD_GAIN / LOAD_MUX"};
            i++;
            while (i < e && g.ops[i].op == OP_BIQUADS) {
                for (int k = 0; k < g.ops[i].n; k++) {
                    secOff.push_back(g.ops[i].a + 6 * k);
                    cols.push_back(g.ops[i].c + 5 * L->nFreq * k);
                    for (int q = 0; q < 5; q++) coefs.push_back(g.pool[g.ops[i].b + 5 * k + q]);
                }
                i++;
            }
            if (i < e && g.ops[i].op == OP_STORE_MEM) {
                // producer half of such a cascade: no output of its own
                if (g.h.aluClass != ALU_INT64 || secOff.empty() || d.srcKind == SRC_LOAD_MUX || findProducer(g.ops[i].a) || (int)producers.size() >= kMaxMemCopy)
                    throw ChainFail{"STORE_MEM the chain kernels cannot inline"};
                MemProducer pr{d.srcKind, d.srcCh, d.srcArg, 0, secOff, coefs, cols};
                producers.emplace_back(g.ops[i].a, pr);
                i++;
                continue;
            }
            d.coefOff = c.h.nPool;
            for (int32_t v : coefs) chainPool(c, v);
            d.secStateOff = c.h.nPool;
            for (int v : secOff) chainPool(c, v);
            d.coefColOff = c.h.nPool;
            for (int v : cols) chainPool(c, v);
            d.nsec = (int16_t)secOff.size();
            if (i < e && g.ops[i].op == OP_GAIN) { d.hasGain = 1; d.gainBits = g.ops[i].a; i++; }
            if (i + 1 < e && g.ops[i].op == OP_DELAY && !d.hasGain && d.nsec > 0 && g.h.aluClass == ALU_INT64 &&
                (g.ops[i + 1].op == OP_SAT0DB || g.ops[i + 1].op == OP_SAT0DB_TPDF || g.ops[i + 1].op == OP_SAT0DB_GAIN || g.ops[i + 1].op == OP_SAT0DB_TPDF_GAIN)) {
                // cascade -> DELAY -> saturation: the delay ring stores (int)X, the low word of the Q59 accumulator, and hands it
                // back sign-extended (dsp_runtime.c:769-794); the saturation stage then works on that
                d.delayOff = g.ops[i].a; d.delayN = g.ops[i].b; d.delayFirst = 1; c.h.nDelayFirst++; i++;
            }
            if (i >= e) throw ChainFail{"a signal path ends without saturation/store"};
            switch (g.ops[i].op) {
            case OP_SAT0DB:           d.satKind = SAT_PLAIN; break;
            case OP_SAT0DB_TPDF:      d.satKind = SAT_TPDF; break;
            case OP_SAT0DB_GAIN:      d.satKind = SAT_GAIN; d.satGainBits = g.ops[i].a; break;
            case OP_SAT0DB_TPDF_GAIN: d.satKind = SAT_TPDF_GAIN; d.satGainBits = g.ops[i].a; break;
            default: throw ChainFail{"a signal path has an opcode the chain kernel does not fuse"};
            }
            i++;
            if (i < e && g.ops[i].op == OP_DELAY && !d.delayFirst) { d.delayOff = g.ops[i].a; d.delayN = g.ops[i].b; i++; }
            if (i >= e || g.ops[i].op != OP_STORE) throw ChainFail{"a signal path does not end with STORE"};
            while (i < e && g.ops[i].op == OP_STORE) {
                if (d.nStores >= kMaxChainStores) throw ChainFail{"too many STOREs on one path"};
                int ch = outChOfSlot[g.ops[i].a];
                if (ch < 0) throw ChainFail{"STORE to a slot outside the declared outputs"};
                claimOutput(ch, d);
                i++;
            }
            if (d.nsec > c.h.maxSec) c.h.maxSec = d.nsec;
            c.h.totalSec += d.nsec;
            c.h.nChains++;
        }
    }
    if (c.h.nChains == 0) throw ChainFail{"no signal path"};
    for (auto& pr : producers) {
        if (pr.second.consumers == 0) throw ChainFail{"a STORE_MEM cascade nobody loads"};
        c.h.memCopyDst[c.h.nMemCopy] = pr.first; c.h.memCopySrc[c.h.nMemCopy] = pr.second.secOff.back(); c.h.nMemCopy++;
    }
    c.h.tpdfShift = kMant - c.h.storeDither + 1;
    // deduplicate the sources of chains that have sections: crossovers feed several cascades from the same
    // LOAD_GAIN (same input, same gain), so their x values are computed and staged once per frame
    c.h.nSrc = 0;
    for (int i = 0; i < c.h.nChains; i++) {
        ChainDesc& d = c.chains[i];
        d.srcId = -1;
        if (d.nsec == 0) continue;
        if (d.srcKind != SRC_LOAD_MUX)
            for (int k = 0; k < c.h.nSrc && d.srcId < 0; k++) {
                const ChainDesc& o = c.chains[c.h.srcChain[k]];
                if (o.srcKind == d.srcKind && o.srcCh == d.srcCh && (d.srcKind == SRC_LOAD || o.srcArg == d.srcArg)) d.srcId = k;
            }
        if (d.srcId < 0) { d.srcId = c.h.nSrc; c.h.srcChain[c.h.nSrc++] = i; }
    }
    c.h.nUnwritten = 0;
    for (int k = 0; k < kIoSlots; k++) {
        c.h.outOff[k] = 0;
        if (k < c.h.nOut) {
            if (c.h.chainOfOut[k] < 0) c.h.nUnwritten++;
            else { const ChainDesc& d = c.chains[c.h.chainOfOut[k]]; c.h.outOff[k] = (d.nsec > 0 ? d.nsec - 1 : 0) - d.delayN; }
        }
    }
    // "direct" chains: cascade -> SAT0DB.  The cascade output is already clamped to [-2^59, 2^59) by the
    // per-section saturation, so dspSaturate64_031 reduces to acc>>28 == the tail section's y1.
    c.h.nAcc = c.h.nProc = 0;
    for (int i = 0; i < c.h.nChains; i++) {
        ChainDesc& d = c.chains[i];
        const bool direct = d.nsec > 0 && !d.hasGain && d.satKind == SAT_PLAIN && !d.delayFirst;
        // (the float class needs no 64-bit accumulator ring: its tails leave the float accumulator in the post ring)
        d.accRow = (d.nsec > 0 && !direct && c.h.aluClass == ALU_INT64) ? c.h.nAcc++ : -1;
        if (!direct) c.h.procChain[c.h.nProc++] = i;
    }
    for (int k = 0; k < kFastTab; k++) {
        c.h.pChain[k] = c.h.pLag[k] = c.h.pFlags[k] = c.h.pGain[k] = c.h.pSatGain[k] = c.h.pDelayN[k] = 0; c.h.pAccRow[k] = -1;
        c.h.sKind[k] = c.h.sArg[k] = 0; c.h.sCh[k] = -1;
        if (k < c.h.nProc) {
            const ChainDesc& d = c.chains[c.h.procChain[k]];
            c.h.pChain[k] = c.h.procChain[k]; c.h.pLag[k] = d.nsec > 0 ? d.nsec - 1 : 0; c.h.pAccRow[k] = d.accRow;
            c.h.pFlags[k] = (d.nsec > 0 ? PF_SECTIONS : 0) | (d.hasGain ? PF_GAIN : 0) | ((d.satKind & 1) ? PF_SAT_TPDF : 0) | (d.satKind >= SAT_GAIN ? PF_SAT_GAIN : 0) |
                            (d.srcKind == SRC_RAW ? PF_RAW : 0);
            if (d.delayFirst) c.h.pFlags[k] = PF_SECTIONS | PF_DELAY_FIRST;      // stage A only parks the accumulator's low word; the sink's stage B finishes
            c.h.pGain[k] = d.gainBits; c.h.pSatGain[k] = d.satGainBits; c.h.pDelayN[k] = d.delayN;
        }
        if (k < c.h.nSrc) {
            const ChainDesc& d = c.chains[c.h.srcChain[k]];
            c.h.sKind[k] = d.srcKind; c.h.sCh[k] = d.srcCh; c.h.sArg[k] = d.srcArg;
        }
    }
}


// ---- DAG recognition (kernel_dag.cu): symbolic execution of the X/Y register pair ------------------------------
namespace {
struct SymVal {
    enum Type { UNDEF = 0, EXPR, FINISHED } type = UNDEF;
    DagOperand a{}, b{};
    int comb = 0, postShift = 0, hasPostGain = 0, postGain = 0;
    int fresh = -1;          // EXPR that is exactly the 64-bit value of this node, nothing applied since
    int node = -1;           // FINISHED: the node whose s.31 output this is
    bool plainOperand() const { return type == EXPR && comb == 0 && postShift == 0 && !hasPostGain; }
};
DagOperand opdNone() { DagOperand o{}; o.kind = OPD_NONE; o.muxStateOff = -1; return o; }
int dagPool(DagPlan& d, int32_t v) {
    if (d.nPool >= kMaxDagPool) throw ChainFail{"DAG pool full"};
    d.pool[d.nPool] = v; return d.nPool++;
}
} // namespace

void buildDagPlan(Lowered* L) {
    const GenericPlan& g = L->gen;
    if (g.h.aluClass != ALU_INT64 || !g.h.sampleInt) throw ChainFail{"the DAG kernel is fixed point (DSP_FORMAT 2)"};
    std::shared_ptr<DagPlan> dp(new DagPlan);
    DagPlan& d = *dp;
    memset(&d, 0, sizeof d);
    d.nIn = g.h.nIn; d.nOut = g.h.nOut;
    d.dataSize = g.h.dataSize; d.stateWords = g.h.stateWords; d.auxOff = g.h.auxOff;
    d.storeDither = g.h.defaultDither;
    for (int k = 0; k < kIoSlots; k++) { d.outNode[k] = -1; d.outDelayed[k] = 0; d.outRaw[k] = -1; }
    int inChOfSlot[kIoSlots], outChOfSlot[kIoSlots];
    for (int k = 0; k < kIoSlots; k++) inChOfSlot[k] = outChOfSlot[k] = -1;
    for (int k = 0; k < g.h.nIn; k++)  inChOfSlot[g.h.inIdx[k]] = k;
    for (int k = 0; k < g.h.nOut; k++) outChOfSlot[g.h.outIdx[k]] = k;
    uint32_t written = 0;
    for (int i = 0; i < g.h.nOps; i++) {
        const MicroOp& m = g.ops[i];
        if (m.op == OP_STORE || m.op == OP_DISTRIB) written |= 1u << m.a;
        if (m.op == OP_LOAD_STORE) for (int k = 0; k < m.n; k++) written |= 1u << g.pool[m.a + 2 * k + 1];
    }
    auto inputCh = [&](int slot) -> int {
        if ((written >> slot) & 1u) throw ChainFail{"an input slot is also written by the program (io hand-off between paths)"};
        return inChOfSlot[slot];             // -1: never fed by the host, reads 0
    };
    std::vector<bool> sealed(kMaxDagNodes, false);     // no more sections may be appended (somebody holds the node's value)
    std::map<int, int> memNode;                        // MEM state offset -> the node stored there last
    auto newNode = [&](const SymVal& in) -> int {
        if (d.nNodes >= kMaxDagNodes) throw ChainFail{"more DAG nodes than kMaxDagNodes"};
        DagNode& n = d.nodes[d.nNodes];
        memset(&n, 0, sizeof n);
        n.a = in.a; n.b = in.comb ? in.b : opdNone();
        n.comb = in.comb; n.postShift = in.postShift; n.hasPostGain = in.hasPostGain; n.postGain = in.postGain;
        n.memOff = -1; n.finKind = FIN_NONE;
        int depth = 0;
        for (const DagOperand* o : {&n.a, &n.b})
            if (o->kind == OPD_NODE) { d.nodes[o->arg].exportAcc = 1; sealed[o->arg] = true; depth = std::max(depth, d.nodes[o->arg].depth + 1); }
        n.depth = depth;
        d.maxDepth = std::max(d.maxDepth, depth);
        return d.nNodes++;
    };
    auto exprOfNode = [&](int id) { SymVal v; v.type = SymVal::EXPR; v.a = opdNone(); v.a.kind = OPD_NODE; v.a.arg = id; v.b = opdNone(); v.fresh = id; return v; };
    auto claimOutput = [&](int ch, int node, int delayed) {
        const int prev = d.outNode[ch];
        if (prev >= 0) {                                // a later STORE of the frame wins: the earlier one is dead
            DagNode& o = d.nodes[prev];
            int w = 0;
            for (int k = 0; k < o.nStores; k++) if (o.storeCh[k] != ch) { o.storeCh[w] = o.storeCh[k]; o.storeDelayed[w] = o.storeDelayed[k]; w++; }
            o.nStores = w;
        }
        d.outNode[ch] = node; d.outDelayed[ch] = delayed; d.outRaw[ch] = -1;
        if (node >= 0) {
            DagNode& n = d.nodes[node];
            if (n.nStores >= kMaxDagStores) throw ChainFail{"too many STOREs on one path"};
            n.storeCh[n.nStores] = ch; n.storeDelayed[n.nStores] = delayed; n.nStores++;
        }
    };
    bool anyXY = false;
    for (int core = 0; core < g.h.nCores; core++) {
        SymVal X, Y;                                     // every core call starts with X = Y = 0 (dsp_runtime.c:308-309)
        X.type = Y.type = SymVal::EXPR; X.a = Y.a = opdNone(); X.b = Y.b = opdNone();
        for (int i = g.h.coreStart[core]; i < g.h.coreStart[core + 1]; i++) {
            const MicroOp& m = g.ops[i];
            switch (m.op) {
            case OP_TPDF_CALC:
                if (core != 0 || d.hasTpdfCalc || d.nNodes) throw ChainFail{"TPDF_CALC not at the very start of core 1"};
                for (int k = 0; k < d.nOut; k++) if (d.outNode[k] != -1) { /* raw copies in front are fine: they use neither the value nor the mask */ }
                d.hasTpdfCalc = 1; d.tpdfDither = m.a; d.tpdfDataOff = m.b; d.storeDither = m.a;
                X = SymVal(); X.type = SymVal::UNDEF;     // X = the dither value: nobody may use it
                break;
            case OP_LOAD_STORE:
                for (int k = 0; k < m.n; k++) {
                    const int ch = outChOfSlot[g.pool[m.a + 2 * k + 1]];
                    if (ch < 0) throw ChainFail{"LOAD_STORE to a slot outside the declared outputs"};
                    claimOutput(ch, -2, 0);
                    d.outNode[ch] = -2; d.outRaw[ch] = inputCh(g.pool[m.a + 2 * k]);
                }
                break;
            case OP_LOAD: case OP_LOAD_GAIN: case OP_LOAD_MUX: {
                Y = X;
                if (Y.fresh >= 0) sealed[Y.fresh] = true;
                X = SymVal(); X.type = SymVal::EXPR; X.a = opdNone(); X.b = opdNone();
                if (m.op == OP_LOAD_MUX) {
                    X.a.kind = OPD_MUX; X.a.n = m.n; X.a.muxStateOff = m.b; X.a.arg = d.nPool;
                    for (int k = 0; k < m.n; k++) { dagPool(d, inputCh(g.pool[m.a + 2 * k])); dagPool(d, g.pool[m.a + 2 * k + 1]); }
                } else {
                    X.a.kind = OPD_RAW; X.a.arg = inputCh(m.a);
                    if (m.op == OP_LOAD_GAIN) { X.a.hasGain = 1; X.a.gain = m.b; }
                }
                break; }
            case OP_LOAD_MEM: {
                Y = X;
                if (Y.fresh >= 0) sealed[Y.fresh] = true;
                auto it = memNode.find(m.a);
                if (it == memNode.end()) throw ChainFail{"LOAD_MEM of a word no earlier path of the frame stored"};
                X = exprOfNode(it->second); X.fresh = -1;           // a copy of the node's value, not the running accumulator
                sealed[it->second] = true;
                break; }
            case OP_STORE_MEM:
                if (X.type != SymVal::EXPR || X.fresh < 0 || !X.plainOperand()) throw ChainFail{"STORE_MEM of something that is not a cascade's accumulator"};
                if (d.nodes[X.fresh].memOff >= 0 && d.nodes[X.fresh].memOff != m.a) throw ChainFail{"one accumulator stored to two MEM words"};
                d.nodes[X.fresh].memOff = m.a; d.nodes[X.fresh].exportAcc = 1; sealed[X.fresh] = true;
                memNode[m.a] = X.fresh;
                break;
            case OP_COPYXY: Y = X; if (X.fresh >= 0) sealed[X.fresh] = true; anyXY = true; break;
            case OP_COPYYX: X = Y; if (Y.fresh >= 0) sealed[Y.fresh] = true; anyXY = true; break;
            case OP_SWAPXY: std::swap(X, Y); anyXY = true; break;
            case OP_CLRXY:  X = SymVal(); X.type = SymVal::EXPR; X.a = opdNone(); X.b = opdNone(); Y = X; break;
            case OP_ADDXY: case OP_SUBXY: case OP_ADDYX: case OP_SUBYX: {
                anyXY = true;
                SymVal& dst = (m.op == OP_ADDXY || m.op == OP_SUBXY) ? X : Y;
                SymVal& src = (m.op == OP_ADDXY || m.op == OP_SUBXY) ? Y : X;
                if (!dst.plainOperand() || !src.plainOperand()) throw ChainFail{"X/Y arithmetic on values the DAG kernel cannot combine"};
                if (dst.a.kind == OPD_NONE && (m.op == OP_ADDXY || m.op == OP_ADDYX)) { const int f = src.fresh; dst = src; dst.fresh = -1; if (f >= 0) sealed[f] = true; break; }
                SymVal r; r.type = SymVal::EXPR; r.a = dst.a; r.b = src.a; r.comb = (m.op == OP_ADDXY || m.op == OP_ADDYX) ? 1 : -1;
                for (const DagOperand* o : {&r.a, &r.b}) if (o->kind == OPD_NODE) sealed[o->arg] = true;
                if (r.b.kind == OPD_NONE) { r.comb = 0; }
                dst = r;
                break; }
            case OP_GAIN:
                if (X.type != SymVal::EXPR) throw ChainFail{"GAIN on a value that is not in the ALU as an expression"};
                if (X.plainOperand() && X.a.kind == OPD_RAW && !X.a.hasGain) { X.a.hasGain = 1; X.a.gain = m.a; }
                else if (!X.hasPostGain && X.a.kind != OPD_NONE) { X.hasPostGain = 1; X.postGain = m.a; }
                else throw ChainFail{"two gains in a row on one value"};
                break;
            case OP_SHIFT: {
                const int sh = m.a <= -100 ? kMant : -m.a;
                if (X.type != SymVal::EXPR || m.a >= 0 || sh > 63 || X.hasPostGain || X.postShift || X.a.kind == OPD_NONE) throw ChainFail{"SHIFT form the DAG kernel does not fuse"};
                if (X.fresh >= 0) sealed[X.fresh] = true;
                X.postShift = sh; X.fresh = -1;
                break; }
            case OP_DELAY:
                if (X.type == SymVal::FINISHED) {
                    DagNode& n = d.nodes[X.node];
                    if (n.delayN) throw ChainFail{"two delays behind one saturation"};
                    n.delayN = m.b; n.delayOff = m.a;
                } else if (X.plainOperand() && X.a.kind == OPD_RAW && !X.a.hasGain && !X.a.delayKind) {
                    X.a.delayKind = 1; X.a.delayN = m.b; X.a.delayOff = m.a;
                } else throw ChainFail{"DELAY on a value the DAG kernel cannot delay (only raw samples and saturated outputs)"};
                break;
            case OP_DELAY_DP:
                if (X.plainOperand() && X.a.kind == OPD_NODE && !X.a.delayKind) {
                    sealed[X.a.arg] = true;
                    X.a.delayKind = 2; X.a.delayN = m.b; X.a.delayOff = m.a; X.fresh = -1;
                } else throw ChainFail{"DELAY_DP on a value the DAG kernel cannot delay (only cascade accumulators)"};
                break;
            case OP_BIQUADS: {
                if (X.type != SymVal::EXPR) throw ChainFail{"BIQUADS on a value that is not in the ALU as an expression"};
                // a lane holds at most 8 sections: longer cascades continue in another node (x = the previous node's value >> 28,
                // which is the previous section's y: exactly what consecutive sections hand to each other)
                for (int first = 0; first < m.n;) {
                    int id;
                    if (X.fresh >= 0 && X.plainOperand() && !sealed[X.fresh] && d.nodes[X.fresh].finKind == FIN_NONE && d.nodes[X.fresh].nsec < 8) id = X.fresh;
                    else { id = newNode(X); d.nodes[id].coefOff = d.nPool; d.nodes[id].secStateOff = -1; }
                    DagNode& n = d.nodes[id];
                    const int take = std::min(m.n - first, 8 - n.nsec);
                    // coefficients and state offsets of a node are contiguous in the pool: re-pack when sections are appended
                    std::vector<int32_t> coefs, offs, cols;
                    for (int k = 0; k < n.nsec; k++) {
                        for (int q = 0; q < 5; q++) coefs.push_back(d.pool[n.coefOff + 5 * k + q]);
                        offs.push_back(d.pool[n.secStateOff + k]); cols.push_back(d.pool[n.coefColOff + k]);
                    }
                    for (int k = first; k < first + take; k++) {
                        for (int q = 0; q < 5; q++) coefs.push_back(g.pool[m.b + 5 * k + q]);
                        offs.push_back(m.a + 6 * k); cols.push_back(m.c + 5 * L->nFreq * k);
                    }
                    n.nsec = (int)offs.size();
                    n.coefOff = d.nPool; for (int32_t v : coefs) dagPool(d, v);
                    n.secStateOff = d.nPool; for (int32_t v : offs) dagPool(d, v);
                    n.coefColOff = d.nPool; for (int32_t v : cols) dagPool(d, v);
                    d.maxSec = std::max(d.maxSec, n.nsec);
                    X = exprOfNode(id);
                    first += take;
                }
                break; }
            case OP_SAT0DB: case OP_SAT0DB_TPDF: case OP_SAT0DB_GAIN: case OP_SAT0DB_TPDF_GAIN: {
                if (X.type != SymVal::EXPR) throw ChainFail{"saturation of a value that is not in the ALU as an expression"};
                int id;
                if (X.fresh >= 0 && X.comb == 0 && X.postShift == 0 && d.nodes[X.fresh].finKind == FIN_NONE) {
                    id = X.fresh;                        // [GAIN] behind the cascade belongs to the finish
                    d.nodes[id].finHasGain = X.hasPostGain; d.nodes[id].finGain = X.postGain;
                } else { SymVal in = X; id = newNode(in); d.nodes[id].nsec = 0; }
                DagNode& n = d.nodes[id];
                n.finKind = FIN_SAT;
                n.satKind = m.op == OP_SAT0DB ? SAT_PLAIN : m.op == OP_SAT0DB_TPDF ? SAT_TPDF : m.op == OP_SAT0DB_GAIN ? SAT_GAIN : SAT_TPDF_GAIN;
                n.satGain = m.a;
                sealed[id] = true;
                X = SymVal(); X.type = SymVal::FINISHED; X.node = id;
                break; }
            case OP_STORE: {
                const int ch = outChOfSlot[m.a];
                if (ch < 0) throw ChainFail{"STORE to a slot outside the declared outputs"};
                if (X.type == SymVal::EXPR) {            // DSP_STORE of an unsaturated value: its low word, masked
                    if (X.a.kind == OPD_NONE && X.comb == 0) throw ChainFail{"STORE of a cleared ALU"};
                    SymVal in = X;
                    const int id = newNode(in);
                    d.nodes[id].nsec = 0; d.nodes[id].finKind = FIN_TRUNC; sealed[id] = true;
                    if (X.fresh >= 0) sealed[X.fresh] = true;
                    X = SymVal(); X.type = SymVal::FINISHED; X.node = id;
                }
                if (X.type != SymVal::FINISHED) throw ChainFail{"STORE of an undefined value"};
                claimOutput(ch, X.node, d.nodes[X.node].delayN > 0 ? 1 : 0);
                break; }
            default:
                throw ChainFail{"an opcode the DAG kernel does not fuse"};
            }
        }
    }
    if (d.nNodes == 0) throw ChainFail{"no signal path"};
    int finals = 0;
    for (int k = 0; k < d.nNodes; k++) {
        const DagNode& n = d.nodes[k];
        if (n.finKind == FIN_NONE && !n.exportAcc) throw ChainFail{"a cascade whose result nobody uses"};
        if (n.finKind != FIN_NONE) finals++;
        for (const DagOperand* o : {&n.a, &n.b}) if (o->kind == OPD_RAW && o->arg >= d.nIn) throw ChainFail{"bad input channel"};
    }
    (void)finals; (void)anyXY;
    d.tpdfShift = kMant - d.storeDither + 1;
    L->dag = dp;
}

// ---- FIR path recognition (kernel_fir.cu) ---------------------------------------------------------
// LOAD|LOAD_GAIN -> FIR(convolution) -> [GAIN] -> SAT0DB|SAT0DB_GAIN -> STORE+ , any number of such paths per core.
void buildFirPlan(Lowered* L) {
    const GenericPlan& g = L->gen;
    FirPlan& f = L->fir;
    memset(&f, 0, sizeof f);
    f.aluClass = g.h.aluClass; f.nIn = g.h.nIn; f.nOut = g.h.nOut; f.stateWords = g.h.stateWords;
    f.storeMask = (int32_t)(0xFFFFFFFFu << ((32 - g.h.defaultDither) & 31));     // dspTpdfPrepare, dsp_tpdf.h:55-80
    if (L->firs.empty()) throw ChainFail{"no DSP_FIR in the program"};
    if (g.h.aluClass == ALU_F64 || !g.h.sampleInt) throw ChainFail{"FIR kernels cover DSP_FORMAT 2 and 3; formats 4..6 run on the generic executor"};
    int inChOfSlot[kIoSlots], outChOfSlot[kIoSlots], owner[kIoSlots];
    for (int k = 0; k < kIoSlots; k++) { inChOfSlot[k] = outChOfSlot[k] = -1; owner[k] = -1; }
    for (int k = 0; k < g.h.nIn; k++)  inChOfSlot[g.h.inIdx[k]] = k;
    for (int k = 0; k < g.h.nOut; k++) outChOfSlot[g.h.outIdx[k]] = k;
    uint32_t written = 0;
    for (int i = 0; i < g.h.nOps; i++) if (g.ops[i].op == OP_STORE) written |= 1u << g.ops[i].a;
    for (int core = 0; core < g.h.nCores; core++) {
        int i = g.h.coreStart[core]; const int e = g.h.coreStart[core + 1];
        while (i < e) {
            if (f.nPaths >= kMaxFirPaths) throw ChainFail{"more than kMaxFirPaths FIR paths"};
            FirPath& d = f.paths[f.nPaths];
            const MicroOp& s = g.ops[i];
            if (s.op != OP_LOAD && s.op != OP_LOAD_GAIN) throw ChainFail{"a path does not start with LOAD / LOAD_GAIN"};
            if ((written >> s.a) & 1u) throw ChainFail{"an input slot is also written by the program"};
            d.srcKind = s.op == OP_LOAD ? SRC_LOAD : SRC_LOAD_GAIN; d.srcCh = inChOfSlot[s.a]; d.srcArg = s.b;
            i++;
            if (i >= e || g.ops[i].op != OP_FIR || g.ops[i].n != 1) throw ChainFail{"a path has no FIR convolution right after its load"};
            d.stateOff = g.ops[i].a; d.tapsOff = g.ops[i].b; d.length = g.ops[i].c; d.tapCol = L->firColOfOp[i];
            if (d.length > kMaxFirTaps) throw ChainFail{"impulse longer than kMaxFirTaps"};
            if (g.h.aluClass == ALU_F32) {
                // the float kernels multiply with mul.rz.ftz.f32, which equals the reference's dspMulFloatFloat (dsp_ieee754.h:336-375)
                // except for products next to 2^-126 (the reference flushes one binade earlier).  |x| >= 2^-31 * |gain| for s.31
                // samples, so with |tap| >= 2^-60 and |gain| >= 2^-30 no product can get there; anything smaller (but non-zero)
                // sends the program to the interpreter, which restates the reference's multiply bit by bit
                auto tiny = [](int32_t bits, int minExp) { const int e = (int)(((uint32_t)bits >> 23) & 255u); return e != 0 && e < 127 + minExp; };
                for (int k = 0; k < d.length; k++)
                    if (tiny(L->bigPool[d.tapsOff + k], -60)) throw ChainFail{"a float tap is smaller than 2^-60: kept on the interpreter for exact underflow behaviour"};
                if (d.srcKind == SRC_LOAD_GAIN && tiny(d.srcArg, -30)) throw ChainFail{"LOAD_GAIN gain smaller than 2^-30 in front of a float FIR"};
            }
            if (d.length > f.maxLen) f.maxLen = d.length;
            i++;
            if (i < e && g.ops[i].op == OP_GAIN) { d.flags |= PF_GAIN; d.gainBits = g.ops[i].a; i++; }
            if (i >= e) throw ChainFail{"a path ends without saturation/store"};
            if (g.ops[i].op == OP_SAT0DB_GAIN) { d.flags |= PF_SAT_GAIN; d.satGainBits = g.ops[i].a; }
            else if (g.ops[i].op != OP_SAT0DB) throw ChainFail{"a FIR path has an opcode the FIR kernels do not fuse"};
            i++;
            if (i >= e || g.ops[i].op != OP_STORE) throw ChainFail{"a path does not end with STORE"};
            while (i < e && g.ops[i].op == OP_STORE) {
                if (d.nStores >= kMaxChainStores) throw ChainFail{"too many STOREs on one path"};
                const int ch = outChOfSlot[g.ops[i].a];
                if (ch < 0) throw ChainFail{"STORE to a slot outside the declared outputs"};
                if (owner[ch] >= 0) throw ChainFail{"two paths store to the same output"};
                owner[ch] = f.nPaths;
                d.storeCh[d.nStores++] = ch;
                i++;
            }
            f.nPaths++;
        }
    }
    if (f.nPaths == 0) throw ChainFail{"no signal path"};
    for (int k = 0; k < g.h.nOut; k++) if (owner[k] < 0) f.unwritten[f.nUnwritten++] = k;
}

// Do the two loop orders agree?  Inside one core the op sequence is the same in both; what differs is WHEN a core sees what
// another core left behind.  So: no MEM word, io slot or dither state may cross a core boundary, and what the plugin copies
// in and out per core (its DSP_CORE bitmaps, fresh io[] per core and frame) must cover what the core reads and writes.
void analyseOrder(Lowered* L) {
    const GenericPlan& g = L->gen;
    auto no = [&](const char* why) { L->orderIndependent = false; L->orderWhy = why; };
    L->orderIndependent = true; L->orderWhy.clear();
    if (g.h.nCores <= 1) return;
    int tpdfCore = -1;
    std::map<int, int> memCore;                       // MEM state offset -> the one core that touches it
    int writer[kIoSlots], reader[kIoSlots];
    for (int k = 0; k < kIoSlots; k++) writer[k] = reader[k] = -1;
    uint32_t hostIn = 0;
    for (int k = 0; k < g.h.nIn; k++) hostIn |= 1u << g.h.inIdx[k];
    for (int c = 0; c < g.h.nCores; c++) {
        const uint32_t cin = L->cores[c].usedIn, cout = L->cores[c].usedOut;
        auto rd = [&](int slot) { if (reader[slot] >= 0 && reader[slot] != c) reader[slot] = -2; else if (reader[slot] != -2) reader[slot] = c;
                                  return !((hostIn >> slot) & 1u) || ((cin >> slot) & 1u); };
        auto wr = [&](int slot) { if (writer[slot] >= 0 && writer[slot] != c) writer[slot] = -2; else if (writer[slot] != -2) writer[slot] = c;
                                  return ((cout >> slot) & 1u) != 0; };
        for (int i = g.h.coreStart[c]; i < g.h.coreStart[c + 1]; i++) {
            const MicroOp& m = g.ops[i];
            bool ok = true;
            switch (m.op) {
            case OP_TPDF_CALC:
                if (tpdfCore >= 0 && tpdfCore != c) return no("DSP_TPDF_CALC in more than one core");
                tpdfCore = c;
                if (m.a != g.h.defaultDither && c != 0) return no("DSP_TPDF_CALC switches the dither table in a core other than the first");
                break;
            case OP_LOAD: case OP_LOAD_GAIN: ok = rd(m.a); break;
            case OP_LOAD_MUX: for (int k = 0; k < m.n; k++) ok = rd(g.pool[m.a + 2 * k]) && ok; break;
            case OP_STORE: case OP_DISTRIB: ok = wr(m.a); break;
            case OP_LOAD_STORE: for (int k = 0; k < m.n; k++) { ok = rd(g.pool[m.a + 2 * k]) && ok; ok = wr(g.pool[m.a + 2 * k + 1]) && ok; } break;
            case OP_LOAD_MEM: case OP_STORE_MEM: {
                auto it = memCore.find(m.a);
                if (it == memCore.end()) memCore[m.a] = c; else if (it->second != c) return no("a MEM word is shared between cores");
                break; }
            case OP_LOAD_MEM_DATA: return no("DSP_LOAD_MEM_DATA reads another opcode's data words");
            default: break;
            }
            if (!ok) return no("a core reads or writes an io slot its DSP_CORE bitmaps do not list (the plugin would not copy it)");
        }
    }
    for (int k = 0; k < kIoSlots; k++)
        if (reader[k] != -1 && writer[k] != -1 && (reader[k] == -2 || writer[k] == -2 || reader[k] != writer[k])) return no("an io slot is handed from one core to another");
    if (tpdfCore >= 0)
        for (int c = 0; c < g.h.nCores; c++) {
            if (c == tpdfCore) continue;
            for (int i = g.h.coreStart[c]; i < g.h.coreStart[c + 1]; i++) {
                const int op = g.ops[i].op;
                if (op == OP_SAT0DB_TPDF || op == OP_SAT0DB_TPDF_GAIN || op == OP_DITHER || op == OP_DITHER_NS2 || op == OP_TPDF || op == OP_WHITE)
                    return no("a core uses the dither value another core computes");
            }
        }
}

// The coefficient-table columns (Lowered::coefWords) and the column of every lowered BIQUADS micro-op.  Section s, fs column f,
// coefficient q of the block at word h is word h + 5 + 6f + s * (2 + 6 * nFreq) + q (dsp_runtime.c:827-849), so within a block
// the columns of a section's fs column are consecutive and sections step by 5 * nFreq.
void buildCoefColumns(Ctx& cx) {
    Lowered* L = cx.L;
    const int stride = 2 + 6 * L->nFreq;
    std::vector<int32_t> cw;
    for (const auto& b : cx.biquadBlocks)
        for (int s = 0; s < b.second; s++)
            for (int f = 0; f < L->nFreq; f++)
                for (int q = 0; q < 5; q++) {
                    const int64_t w = (int64_t)b.first + 5 + 6 * f + (int64_t)s * stride + q;
                    if (w >= 0 && w < cx.total) cw.push_back((int32_t)w);
                }
    std::sort(cw.begin(), cw.end());
    cw.erase(std::unique(cw.begin(), cw.end()), cw.end());
    L->coefWords = cw;
    auto colOf = [&](int64_t w) -> int64_t {
        auto it = std::lower_bound(cw.begin(), cw.end(), (int32_t)std::min<int64_t>(w, INT32_MAX));
        return (it != cw.end() && *it == w) ? (int64_t)(it - cw.begin()) : -1;
    };
    L->coefTableOk = true;
    GenericPlan& g = L->gen;
    for (int i = 0; i < g.h.nOps; i++) {
        MicroOp& m = g.ops[i];
        if (m.op != OP_BIQUADS) continue;
        const int64_t c0 = (int64_t)m.c + 5 + 6 * L->fsRel;
        const int64_t col0 = colOf(c0);
        for (int s = 0; s < m.n; s++)
            for (int q = 0; q < 5; q++)
                if (col0 < 0 || colOf(c0 + (int64_t)s * stride + q) != col0 + 5 * L->nFreq * s + q) L->coefTableOk = false;
        m.c = col0 < 0 ? 0 : (int32_t)col0;
    }
}

// The FIR-table columns (Lowered::firTapWords) and the column of every lowered FIR convolution.  A tap block is a run of
// consecutive words, all of them listed, so its taps sit in consecutive columns whatever other blocks overlap it.
void buildFirColumns(Ctx& cx) {
    Lowered* L = cx.L;
    std::vector<int32_t> tw;
    for (const auto& b : cx.firBlocks)
        for (int k = 0; k < b.second && (int64_t)b.first + k < cx.total; k++) tw.push_back(b.first + k);
    std::sort(tw.begin(), tw.end());
    tw.erase(std::unique(tw.begin(), tw.end()), tw.end());
    L->firTapWords = tw;
    L->firColOfOp.assign(cx.firConvs.empty() ? 0 : (size_t)L->gen.h.nOps, -1);
    for (const auto& c : cx.firConvs)
        L->firColOfOp[c.first] = (int32_t)(std::lower_bound(tw.begin(), tw.end(), c.second) - tw.begin());
}

void lowerAll(Lowered* L) {
    Ctx cx; cx.L = L; cx.w = L->words.data(); cx.total = L->totalLength;
    cx.delayFactor = (uint32_t)(4294.967296 * (double)L->fs);      // dsp_runtime.c:81-90
    GenericPlan& g = L->gen;
    const std::vector<int> keepMem = L->memWord;                   // keep slot numbering stable on re-lowering
    L->memWord.clear();
    for (size_t k = 0; k < keepMem.size(); k++) cx.memSlot(keepMem[k], 0);
    g.h.nOps = 0; g.h.nPool = 0;
    L->bigPool.clear(); L->firs.clear(); cx.biquadBlocks.clear(); cx.firBlocks.clear(); cx.firConvs.clear();

    g.h.nCores = (int)L->cores.size();
    uint32_t usedIn = 0, usedOut = 0;
    for (int c = 0; c < g.h.nCores; c++) {
        g.h.coreStart[c] = g.h.nOps;
        lowerCore(cx, L->cores[c].beginWord);
        usedIn |= L->cores[c].usedIn; usedOut |= L->cores[c].usedOut;
    }
    g.h.coreStart[g.h.nCores] = g.h.nOps;
    g.h.nIn = g.h.nOut = 0;
    for (int k = 0; k < kIoSlots; k++) {
        if ((usedIn >> k) & 1u)  g.h.inIdx[g.h.nIn++] = (uint8_t)k;
        if ((usedOut >> k) & 1u) g.h.outIdx[g.h.nOut++] = (uint8_t)k;
    }
    // state block layout
    g.h.dataSize = L->dataSize;
    g.h.auxOff = (L->dataSize + 1) & ~1;
    g.h.memOff = g.h.auxOff + kAuxWords;
    g.h.nMem = cx.nMemSlots;
    g.h.stateWords = (g.h.memOff + 2 * g.h.nMem + 3) & ~3;
    for (int i = 0; i < g.h.nOps; i++)
        if (g.ops[i].op == OP_LOAD_MEM || g.ops[i].op == OP_STORE_MEM) g.ops[i].a = g.h.memOff + 2 * g.ops[i].a;
    buildCoefColumns(cx);
    buildFirColumns(cx);

    analyseOrder(L);
    try { buildChainPlan(L); L->chainOk = true; L->chainWhyNot.clear(); }
    catch (const ChainFail& f) { L->chainOk = false; L->chainWhyNot = f.why; }
    L->dag.reset();
    try { buildDagPlan(L); L->dagOk = true; L->dagWhyNot.clear(); }
    catch (const ChainFail& f) { L->dagOk = false; L->dagWhyNot = f.why; L->dag.reset(); }
    try { buildFirPlan(L); L->firOk = true; L->firWhyNot.clear(); }
    catch (const ChainFail& f) { L->firOk = false; L->firWhyNot = f.why; }

    // lowering trace (the B200 counterpart of the reference's DSP_PRINTF>=2 opcode trace)
    char line[160];
    L->trace.clear();
    for (int c = 0; c < g.h.nCores; c++) {
        snprintf(line, sizeof line, "core %d: ops [%d,%d)\n", c + 1, g.h.coreStart[c], g.h.coreStart[c + 1]); L->trace += line;
        for (int i = g.h.coreStart[c]; i < g.h.coreStart[c + 1]; i++) {
            const MicroOp& m = g.ops[i];
            snprintf(line, sizeof line, "  %3d op=%2d n=%d a=%d b=%d c=%d\n", i, m.op, m.n, m.a, m.b, m.c); L->trace += line;
        }
    }
    L->trace += std::string("loop order: ") + (L->orderIndependent ? "plugin order == canonical order (no data crosses a core boundary)" : ("order-dependent: " + L->orderWhy)) + "\n";
    snprintf(line, sizeof line, "state: data=%d aux@%d mem@%d x%d words/stream=%d; chain kernel: %s%s\n",
             g.h.dataSize, g.h.auxOff, g.h.memOff, g.h.nMem, g.h.stateWords, L->chainOk ? "yes" : "no: ", L->chainWhyNot.c_str());
    L->trace += line;
}

} // namespace

int findCoreWord(const int32_t* prog, int numCore) {
    if (wordOpcode(prog[0]) != OP_HEADER) return -1;
    int p = 0, num = 0;
    for (;;) {
        int sk = wordSkip(prog[p]);
        if (sk == 0) return num == 0 ? 0 : -1;      // no DSP_CORE at all: the program itself (:50-52)
        if (wordOpcode(prog[p]) == OP_CORE && ++num == numCore) return p;
        p += sk;
    }
}

int findCoreBeginWord(const int32_t* prog, int p) {
    if (p < 0 || wordOpcode(prog[p]) != OP_CORE) return p;
    for (;;) {
        int op = wordOpcode(prog[p]), sk = wordSkip(prog[p]);
        if (sk == 0) return p;
        if (op == OP_CORE || op == OP_NOP || op == OP_PARAM || op == OP_PARAM_NUM) p += sk; else return p;
    }
}

int decodeProgram(const int32_t* prog, int progWords, int maxWords, int format, int fs,
                  int defaultDither, Lowered* L, std::string* err) {
    auto bad = [&](int code, const char* msg) { if (err) *err = msg; return code; };
    if (format < FMT_INT64 || format > FMT_DOUBLE_FLOAT) return bad(ERR_FORMAT, "DSP_FORMAT must be 2..6");
    if (!prog || progWords < H_WORDS || wordOpcode(prog[0]) != OP_HEADER) return bad(ERR_NO_HEADER, "no dsp header in this program");
    const int total = prog[H_TOTAL], dsz = prog[H_DATASIZE];
    if (total < H_WORDS || dsz < 0 || total > progWords) return bad(ERR_TOO_LARGE, "header totalLength exceeds the words provided");
    if ((int64_t)total + dsz > (int64_t)maxWords) return bad(ERR_TOO_LARGE, "program+data is over the allowed size");
    // dspCalcSumCore
    uint32_t sum = 0; int ncores = 0, p = 0;
    for (;;) {
        if (p >= total) return bad(ERR_CHECKSUM, "opcode chain runs past totalLength");
        int sk = wordSkip(prog[p]);
        if (sk == 0) { if (ncores == 0) ncores = 1; break; }
        if (wordOpcode(prog[p]) == OP_CORE) ncores++;
        sum += (uint32_t)prog[p];
        p += sk;
    }
    if (ncores < 1) return bad(ERR_NO_CORE, "no cores defined in the program");
    if (sum != (uint32_t)prog[H_CHECKSUM]) return bad(ERR_CHECKSUM, "checksum problem with the program");
    // encoder 0x100 files (module_avdsp/rpi/*.bin, osx/mydspcode.bin: 11-word header, TPDF_CALC without its data word)
    // decode to wild data offsets in the reference runtime itself, which does not look at the version: named error here
    if (wordSkip(prog[0]) != H_WORDS || prog[H_VERSION] < kMinEncoderVersion)
        return bad(ERR_ENCODER_OLD, "program was made by an encoder older than 0x102 (different header / opcode layouts)");
    const int maxOpcode = (int)((uint32_t)prog[H_FORMAT] >> 16), enc = (int)((uint32_t)prog[H_FORMAT] & 0xFFFF);
    if (maxOpcode >= OP_MAX_OPCODE) return bad(ERR_OPCODE_NEW, "program uses opcodes newer than this runtime");
    // The reference converts encodings in place (dspChangeFormat) but that path is unreliable
    // (SURVEY.md App. C #6); we require programs encoded for the format they run in.
    if (format == FMT_INT64 ? enc != kMant : enc != 0) return bad(ERR_FORMAT, "program is not encoded for the requested DSP_FORMAT");
    const int fi = freqToIndex(fs);
    if (fi >= kNumFreq) return bad(ERR_NO_HEADER, "sampling frequency not supported");
    const int fmin = prog[H_FREQMIN], fmax = prog[H_FREQMAX];
    if (fi < fmin || fi > fmax) return bad(ERR_FS_RANGE, "sampling freq not compatible with encoded dsp program");

    *L = Lowered{};
    L->format = format; L->fs = fs; L->fsIndex = fi; L->fsRel = fi - fmin; L->nFreq = fmax - fmin + 1;
    L->totalLength = total; L->dataSize = dsz; L->defaultDither = defaultDither;
    L->words.assign(prog, prog + total);
    L->gen.h.format = format;
    L->gen.h.aluClass = (format == FMT_INT64) ? ALU_INT64 : (format == FMT_FLOAT || format == FMT_FLOAT_FLOAT) ? ALU_F32 : ALU_F64;
    L->gen.h.sampleInt = (format <= FMT_DOUBLE) ? 1 : 0;
    L->gen.h.defaultDither = defaultDither;
    for (int k = 1; k <= kMaxCores + 1; k++) {
        int cw = findCoreWord(prog, k);
        if (cw < 0) break;
        if (k > kMaxCores) return bad(ERR_PLAN_SIZE, "more DSP_CORE sections than the executor supports");
        CoreInfo ci;
        ci.coreWord = cw;
        if (wordOpcode(prog[cw]) == OP_CORE && cw + 2 >= total) return bad(ERR_MALFORMED, "DSP_CORE in the last words of the program");
        if (wordOpcode(prog[cw]) == OP_CORE) { ci.beginWord = findCoreBeginWord(prog, cw); ci.usedIn = (uint32_t)prog[cw + 1]; ci.usedOut = (uint32_t)prog[cw + 2]; }
        else { ci.beginWord = 0; ci.usedIn = (uint32_t)prog[H_USEDIN]; ci.usedOut = (uint32_t)prog[H_USEDOUT]; }
        L->cores.push_back(ci);
        if (wordOpcode(prog[cw]) != OP_CORE) break;     // program without DSP_CORE: exactly one core (not 8x, App. C #8)
    }
    try { lowerAll(L); }
    catch (const Fail& f) { if (err) *err = f.msg; return f.code; }
    return total;
}

int relowerProgram(const int32_t* prog, int progWords, Lowered* L, std::string* err) {
    if (progWords < L->totalLength) { if (err) *err = "fewer words than the loaded program"; return ERR_ARG; }
    // structure (opcode words) must be unchanged: only parameter words may differ
    int p = 0;
    for (;;) {
        if (prog[p] != L->words[p]) { if (err) *err = "opcode structure changed; create a new instance instead"; return ERR_ARG; }
        int sk = wordSkip(prog[p]);
        if (sk == 0) break;
        p += sk;
    }
    // lower into a copy and swap it in only on success: a failure leaves every plan, pool and MEM table as it was
    std::unique_ptr<Lowered> tmp(new Lowered(*L));
    tmp->words.assign(prog, prog + L->totalLength);
    try { lowerAll(tmp.get()); }
    catch (const Fail& f) { if (err) *err = f.msg; return f.code; }
    if (tmp->gen.h.stateWords != L->gen.h.stateWords) { if (err) *err = "state layout changed"; return ERR_ARG; }
    *L = std::move(*tmp);
    return L->totalLength;
}

} // namespace avdsp

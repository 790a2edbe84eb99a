/*
 * avdsp_b200.h -- C ABI of the B200-native batched executor for AVDSP encoded DSP programs.
 *
 * This is the drop-in boundary of the hot path.  Plain pointers and sizes only; no torch/C++
 * types.  Two groups of entry points:
 *
 *  (1) the reference runtime's own entry points, same names, arguments and return codes, so a host
 *      written against /root/reference/module_avdsp/runtime/dsp_runtime.h:160-164 links unchanged
 *      (per-frame compatibility path: every call is a 1-stream, 1-frame launch -- correct but slow);
 *  (2) the batched variant the ALSA host (module_avdsp/linux/avdsp_plugin.c:71-163, dsp_transfer)
 *      calls once per period for all frames -- and for any number of independent streams.
 *
 * All numerics are the reference's: DSP_FORMAT 2 (int64 accumulator) is bit-exact; formats 3..6
 * reproduce the reference's hand-rolled IEEE helpers (runtime/dsp_ieee754.h) bit for bit, in the
 * generic executor and in the fused kernels (formats 3 and 5: hardware multiplies behind a per-stream
 * exactness guard, flagged streams re-executed exactly inside the same call).  The one path with a
 * stated tolerance is the opt-in 3xTF32 tensor-core FIR (AVDSP_B200_KERNEL_FIR_TC on a float program).
 *
 * There is no CPU fallback: every compute entry point returns AVDSP_B200_ERR_CUDA when no CUDA
 * device is usable.
 */
#ifndef AVDSP_B200_H_
#define AVDSP_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------------------------------
 * (1) Reference entry points.  opcode_t is a 32-bit word (runtime/dsp_header.h:197-209) and
 *     dspSample_t is a 32-bit word (int for formats 2..4, float for 5/6; runtime/dsp_runtime.h:51-127),
 *     so both are spelled int32_t / void here.
 * ------------------------------------------------------------------------------------------ */

/* replaces dspRuntimeInit, runtime/dsp_runtime.c:150-195.
 * returns totalLength (>0) or -1 no header, -3 no core, -4 checksum, -5 opcode too recent,
 * -6 program+data larger than maxSize, and dspRuntimeReset's -1/-2 when fs != 0.
 * The executor keeps `codePtr` (one live program per process, like the reference's dspHeaderPtr
 * global, :36,156) and mirrors the data area / MEM words back into the caller's buffer after
 * every dspRuntime_<fmt> call, since reference hosts own and inspect that buffer. */
int  dspRuntimeInit(int32_t *codePtr, int maxSize, const int fs, int random, int defaultDither);
/* replaces dspRuntimeReset, runtime/dsp_runtime.c:116-145.  0 | -1 unknown fs | -2 fs outside header range */
int  dspRuntimeReset(const int fs, int random, int defaultDither);
/* replaces dspFindCore, runtime/dsp_runtime.c:42-59 (numCore is 1-based; 0 when absent) */
int32_t *dspFindCore(int32_t *codePtr, const int numCore);
/* replaces dspFindCoreBegin, runtime/dsp_runtime.c:62-77 */
int32_t *dspFindCoreBegin(int32_t *corePtr);
/* replace dspRuntime_<DSP_FORMAT>, runtime/dsp_runtime.c:302-1314 (name mangling runtime/dsp_runtime.h:41-127,164):
 * run ONE core for ONE frame.  io = the 32-slot sample array.  Always returns 0 like the reference
 * (negative only when no program is loaded or CUDA failed). */
int  dspRuntime_2(int32_t *corePtr, int *rundataPtr, void *io);
int  dspRuntime_3(int32_t *corePtr, int *rundataPtr, void *io);
int  dspRuntime_4(int32_t *corePtr, int *rundataPtr, void *io);
int  dspRuntime_5(int32_t *corePtr, int *rundataPtr, void *io);
int  dspRuntime_6(int32_t *corePtr, int *rundataPtr, void *io);
/* replace dspQNM / dspQM64 / dspQM32, runtime/dsp_header.c:76-86 (macros runtime/dsp_header.h:276-285) */
long long dspQNM(double x, int n, int m);
long long dspQM64(double x, int m);
int       dspQM32(double x, int m);
/* replaces dspOpcodeText, runtime/dsp_header.c:10-73 */
#define AVDSP_B200_MAX_OPCODE 62
extern const char *dspOpcodeText[AVDSP_B200_MAX_OPCODE];

/* ------------------------------------------------------------------------------------------
 * (2) Batched executor.  Replaces the per-period loop nest of dsp_transfer
 *     (module_avdsp/linux/avdsp_plugin.c:95-142): "for core: for frame: gather io, dspRuntime, scatter".
 * ------------------------------------------------------------------------------------------ */
typedef struct avdsp_b200 avdsp_b200_t;

/* error codes: the first six are the reference's (runtime/dsp_runtime.c:116-195) */
enum {
    AVDSP_B200_ERR_NO_HEADER   = -1,   /* also: unknown sampling frequency */
    AVDSP_B200_ERR_FS_RANGE    = -2,
    AVDSP_B200_ERR_NO_CORE     = -3,
    AVDSP_B200_ERR_CHECKSUM    = -4,
    AVDSP_B200_ERR_OPCODE_NEW  = -5,
    AVDSP_B200_ERR_TOO_LARGE   = -6,
    AVDSP_B200_ERR_FORMAT      = -7,   /* unsupported DSP_FORMAT / program encoded for another format */
    AVDSP_B200_ERR_UNSUPPORTED = -8,   /* opcode the executor rejects (DSP_SINE: does not compile in the reference) */
    AVDSP_B200_ERR_ARG         = -9,
    AVDSP_B200_ERR_CUDA        = -10,
    AVDSP_B200_ERR_MALFORMED   = -11,  /* a pointer/offset in the program leaves the program or its data area */
    AVDSP_B200_ERR_PLAN_SIZE   = -12,  /* lowered plan exceeds the kernel-parameter budget */
    AVDSP_B200_ERR_ENCODER_OLD = -13   /* file made by an encoder older than 0x102 (the .bin files under module_avdsp/rpi: 11-word header, TPDF_CALC
                                          without its data word): the reference runtime does not check and walks into wild offsets */
};

/* PCM layouts.  A "frame" is one sample for every channel (one dspRuntime call per core in the reference). */
enum { AVDSP_B200_INTERLEAVED = 0,     /* [stream][frame][channel]  (what ALSA hands to dsp_transfer) */
       AVDSP_B200_PLANAR      = 1 };   /* [stream][channel][frame] */
enum { AVDSP_B200_HOST = 0, AVDSP_B200_DEVICE = 1 };
/* kernel selection (diagnostics and tests; AUTO is the product behaviour) */
enum { AVDSP_B200_KERNEL_AUTO = 0, AVDSP_B200_KERNEL_GENERIC = 1, AVDSP_B200_KERNEL_CHAIN = 2,
       AVDSP_B200_KERNEL_CHAIN_V1 = 3 /* removed (the first, tile-synchronous chain kernel): selecting it returns ERR_UNSUPPORTED */,
       AVDSP_B200_KERNEL_MIX = 4      /* time-parallel kernel for programs without biquads (mixers, delays, dither) */,
       AVDSP_B200_KERNEL_FIR = 5      /* time-parallel tiled DSP_FIR kernels (runtime/dsp_firSTD.h, dsp_runtime.c:928-969) */,
       AVDSP_B200_KERNEL_FIR_TC = 6   /* DSP_FIR as a Toeplitz GEMM on tcgen05 tensor cores: DSP_FORMAT 2 bit-exact (8-bit limbs, the
                                         AUTO choice for batches), DSP_FORMAT 3 as 3xTF32 under a stated tolerance (only on request) */,
       AVDSP_B200_KERNEL_CHAIN_V2 = 7 /* force the section-lane chain kernel (kernel_chain2.cu) */,
       AVDSP_B200_KERNEL_CHAIN_V3 = 8 /* force the cascade-per-lane chain kernel (kernel_chain3.cu); KERNEL_CHAIN / AUTO pick between
                                         v2 and v3 themselves (v3: common crossover / EQ shapes at batch width) */,
       AVDSP_B200_KERNEL_DAG = 9      /* programs that route signals through the X/Y registers (subtractive crossovers, forks, sums of MEM
                                         words): a DAG of cascades, one node per warp (kernel_dag.cu); AUTO takes it when no other fused
                                         kernel can run the program */ };

/* Load + validate + lower a program (dspRuntimeInit + dspRuntimeReset for nStreams independent
 * instances).  prog: progWords little-endian 32-bit words exactly as written by dspcreate (.bin).
 * format: DSP_FORMAT 2..6.  seeds: per-stream dither PRNG seed (`random` of dspRuntimeInit), NULL => 0
 * for every stream (what the ALSA plugin passes, avdsp_plugin.c:178).  device: CUDA ordinal.
 * returns totalLength (>0) or a negative error code. */
int  avdsp_b200_create(avdsp_b200_t **out, const int32_t *prog, int progWords, int fs, int format,
                       int nStreams, const int32_t *seeds, int defaultDither, int device);
/* The same over several GPUs of one box (SURVEY.md 8b `deviceMask`): bit d of deviceMask = CUDA device d takes part.  The
 * streams are cut into contiguous balanced ranges, one per device (the first nStreams mod n ranges one stream longer); each
 * range is an independent single-device instance, no collective on the data path.  A multi-device instance takes HOST
 * buffers only (avdsp_b200_process / _process_pcm / _copy_only with AVDSP_B200_HOST): one call fans the buffer out, one
 * staging thread per GPU running on the host NUMA node next to it.  Everything else (reset, reload_params, set_order,
 * get/set_state by global stream index, io_map, ...) works as on a single-device instance; avdsp_b200_process_async /
 * _process_range return AVDSP_B200_ERR_UNSUPPORTED. */
int  avdsp_b200_create_multi(avdsp_b200_t **out, const int32_t *prog, int progWords, int fs, int format,
                             int nStreams, const int32_t *seeds, int defaultDither, unsigned deviceMask);
int  avdsp_b200_num_devices(const avdsp_b200_t *);
/* shard k of the instance: its CUDA device, stream range and the host NUMA node next to that device (-1: unknown) */
int  avdsp_b200_shard_info(const avdsp_b200_t *, int k, int *device, int *firstStream, int *nStreams, int *numaNode);
/* Page-locked PCM buffer of nStreams * bytesPerStream bytes placed for this instance: every shard's slice (both layouts are
 * stream-major, so a shard's streams are one contiguous slice) lies on the host NUMA node next to the GPU that will DMA
 * it.  The host path works with any host memory; buffers from here are what makes it scale over the GPUs of a box. */
void *avdsp_b200_host_alloc(avdsp_b200_t *, size_t bytesPerStream);
void avdsp_b200_host_free(avdsp_b200_t *, void *p);
void avdsp_b200_destroy(avdsp_b200_t *);
/* dspRuntimeReset for every stream: zero the data area, re-seed the PRNG, MEM words back to the
 * program's initial values.  fs may change (must stay inside the program's range). */
int  avdsp_b200_reset(avdsp_b200_t *, int fs, const int32_t *seeds, int defaultDither);

/* I/O map = union of the DSP_CORE used-input / used-output bitmaps in ascending io-slot order
 * (what avdsp_plugin.c:326-356 derives).  Arrays need room for 32 ints; any pointer may be NULL. */
int  avdsp_b200_io_map(const avdsp_b200_t *, int *nIn, int *inIdx, int *nOut, int *outIdx);

/* Process nFrames frames of every stream.  in: nStreams*nFrames*nIn 32-bit samples, out:
 * nStreams*nFrames*nOut, both in `layout`; memspace says where the two buffers live.  Canonical
 * order (frame-major, cores ascending, one io[] per frame) unless avdsp_b200_set_order chose the
 * plugin's.  Any split of a frame range into successive calls gives identical output. Synchronous. */
int  avdsp_b200_process(avdsp_b200_t *, const void *in, void *out, int nFrames, int layout, int memspace);
/* The DMA schedule of avdsp_b200_process(HOST) without the kernel launches: what the box's PCIe / host memory can do for
 * exactly this call.  bench.py reports e2e against it. */
int  avdsp_b200_copy_only(avdsp_b200_t *, const void *in, void *out, int nFrames, int layout);
/* Same with device buffers, enqueued on the caller's CUDA stream (cudaStream_t as void*), no sync.
 * Calls on ONE instance are stream-ordered by the library whatever stream they are given (each launch waits for the
 * instance's previous launch: launches continue each other's state and share per-instance scratch); instances are
 * independent of each other.  reload_params / reset / get_state / set_state wait for everything launched before. */
int  avdsp_b200_process_async(avdsp_b200_t *, const void *in, void *out, int nFrames, int layout, void *cudaStream);
/* Process a sub-range of the streams: [firstStream, firstStream+nStreams) (buffers hold only those). */
int  avdsp_b200_process_range(avdsp_b200_t *, const void *in, void *out, int nFrames, int layout,
                              int firstStream, int nStreams, void *cudaStream);

/* The ALSA plugin's input formats (linux/avdsp_plugin.c:109-121): interleaved S16_LE / S24_3LE / S32_LE frames are
 * widened to s.31 on the device (S16: <<16; S24_3LE: b0<<8 | b1<<16 | b2<<24), output is always S32 (:138, :364).
 * in: nStreams*nFrames*nIn samples of `pcmFormat`, interleaved; out: nStreams*nFrames*nOut int32. Synchronous. */
enum { AVDSP_B200_PCM_S32 = 0, AVDSP_B200_PCM_S16 = 1, AVDSP_B200_PCM_S24_3LE = 2 };
int  avdsp_b200_process_pcm(avdsp_b200_t *, const void *in, int pcmFormat, void *out, int nFrames, int memspace);

/* period == 0: canonical order.  period > 0: the ALSA plugin's core-major loop nest with this period
 * (avdsp_plugin.c:95-98), fresh io[] per (core, frame). */
int  avdsp_b200_set_order(avdsp_b200_t *, int period);
int  avdsp_b200_set_kernel(avdsp_b200_t *, int which);
/* which kernel the last process call used (AVDSP_B200_KERNEL_*) and how many kernels were launched so far */
int  avdsp_b200_last_kernel(const avdsp_b200_t *);
/* 2 or 3 when the last call ran a chain kernel (which of kernel_chain2.cu / kernel_chain3.cu), else 0 */
int  avdsp_b200_last_chain_variant(const avdsp_b200_t *);
long long avdsp_b200_launch_count(const avdsp_b200_t *);

/* The host edited PARAM words (gains, delay times, biquad coefficients, bypass flags) of the loaded
 * program -- the dump-file workflow, encoder/dsp_encoder.c:476-503.  Opcode structure must be unchanged. */
int  avdsp_b200_reload_params(avdsp_b200_t *, const int32_t *prog, int progWords);

/* Per-stream parameters (the dump-file workflow per stream: a different crossover / EQ / delay / gain per room).
 * From now on the streams [firstStream, firstStream + nStreams) run with the program words [wordIndex, wordIndex + nWords)
 * replaced by `values` (PARAM data: gains, biquad coefficients, delay words, bypass flags ...).  Cumulative per stream;
 * opcode words and the state layout must stay as they are (same rule as avdsp_b200_reload_params, which also clears every
 * override).  Streams keep their state.  Cost model: streams that share one parameter set AND are neighbours run in one
 * launch -- give each room a contiguous stream range.  avdsp_b200_param_index turns a dump-file entry `name offset num size`
 * (encoder/dsp_encoder.c:476-503: offset relative to the data of DSP_PARAM_NUM section `num`, absolute when num == 0) into
 * the word index to pass here. */
int  avdsp_b200_param_index(const avdsp_b200_t *, int offset, int paramNum);
int  avdsp_b200_set_param(avdsp_b200_t *, int firstStream, int nStreams, int wordIndex, const int32_t *values, int nWords);
int  avdsp_b200_num_variants(const avdsp_b200_t *);      /* distinct parameter sets alive (1 = no override) */

/* Per-stream biquad coefficients in one launch: a room EQ or crossover per stream without a parameter variant per stream.
 *
 * Program words that are biquad coefficients: the b0 b1 b2 a1 a2 words of every section of every DSP_BIQUADS parameter block,
 * for EVERY sampling-frequency column, bypassed blocks included.  Listed once each, in ascending word order (two BIQUADS opcodes
 * that share a parameter block share its words).  The list is the column order of avdsp_b200_set_coefs.  Host-only: validates
 * the program like avdsp_b200_describe (same error codes) and needs no instance and no CUDA device.  Writes at most maxOut
 * indices and returns the count (0: no biquad in the program), or an error code. */
int  avdsp_b200_coef_words(const int32_t *prog, int progWords, int format, int32_t *wordIndex, int maxOut);
/* Per-stream coefficients at batch width.  values = nStreams rows of nCoef 32-bit words, nCoef = the count avdsp_b200_coef_words
 * returns; row s holds the coefficient words of stream firstStream + s in that column order: Q4.28 integers for DSP_FORMAT 2,
 * float bit patterns for the float formats.  memspace AVDSP_B200_HOST: the rows are copied before the call returns.
 * AVDSP_B200_DEVICE: the buffer is read in order on cudaStream (a cudaStream_t), after every launch enqueued on the instance
 * before this call, and the host is not blocked (the first call of an instance allocates the table and may wait).
 * The effect is exactly avdsp_b200_set_param(firstStream + s, 1, w, &row[s][col], 1) for every stream s and column col with word
 * index w, and outputs and state are bit-identical to that; but a call still costs the launches of one parameter set, however
 * many distinct rows there are (the kernels load each stream's coefficients from the table once per launch).
 *  - The first call creates the instance's coefficient table.  Every stream's row starts from the words the stream runs with at
 *    that moment: the program's, or those of its set_param variant.  avdsp_b200_num_variants does not count the table.
 *  - The latest call wins for a word.  While a table exists, set_param on coefficient words writes those streams' rows and
 *    creates no variant; set_param on any other word (gains, delays, bypass flags) makes variants as before, and they combine
 *    with the rows.  Runs of neighbouring streams that share a variant launch as before, every launch reading the table.
 *  - reload_params drops the table (like every override).  reset keeps it: rows hold every fs column, so a reset to another
 *    rate runs that rate's columns.
 *  - Refusals change nothing: AVDSP_B200_ERR_UNSUPPORTED for a program without biquad coefficients, for DEVICE rows on a
 *    multi-device instance (HOST rows are split over its shards), and for a program whose parameter blocks overlap or a variant
 *    that changed a block's section count; AVDSP_B200_ERR_ARG for a bad stream range, NULL values or an unknown memspace.
 *  - DSP_FORMAT 3 and 5 on the chain kernels: a row with a non-zero coefficient outside [2^-60, 2^7) sends its stream through the
 *    exact re-execution of the float class inside the same call, so every stream stays bit-exact. */
int  avdsp_b200_set_coefs(avdsp_b200_t *, int firstStream, int nStreams, const int32_t *values, int memspace, void *cudaStream);

/* Per-stream FIR taps in one launch: a room-correction impulse response per stream without a parameter variant per stream.
 * The rules are those of the biquad coefficient table above; the two tables are independent and may coexist.
 *
 * Program words that are FIR taps: for every DSP_FIR opcode and EVERY sampling-frequency column whose entry is a convolution
 * (length word lw > 0 with lw >> 16 == 0), the words t + 1 .. t + lw after its length word t.  Plain-delay entries
 * (lw >> 16 != 0) and skipped entries (relative pointer 0) contribute nothing.  Listed once each, in ascending word order (two
 * opcodes that point at one tap block share its words).  The list is the column order of avdsp_b200_set_fir_taps.  Host-only:
 * validates the program like avdsp_b200_describe at EVERY rate it admits (same error codes) and needs no instance and no CUDA
 * device.  Writes at most
 * maxOut indices and returns the count (0: no FIR convolution in the program), or an error code. */
int  avdsp_b200_fir_tap_words(const int32_t *prog, int progWords, int format, int32_t *wordIndex, int maxOut);
/* Per-stream taps at batch width.  values = nStreams rows of nTaps 32-bit words, nTaps = the count avdsp_b200_fir_tap_words
 * returns; row s holds the tap words of stream firstStream + s in that column order: Q4.28 integers for DSP_FORMAT 2, float bit
 * patterns for the float formats.  memspace AVDSP_B200_HOST: the rows are copied before the call returns.  AVDSP_B200_DEVICE:
 * the buffer is read in order on cudaStream (a cudaStream_t), after every launch enqueued on the instance before this call, and
 * the host is not blocked (the first call of an instance allocates the table and may wait).
 * The effect is exactly avdsp_b200_set_param(firstStream + s, 1, w, &row[s][col], 1) for every stream s and column col with word
 * index w, and outputs and state are bit-identical to that; but a call still costs the launches of one parameter set, however
 * many distinct rows there are (the FIR kernels stage each stream's taps from its row).
 *  - The table holds nStreams x nTaps words on the device (C4, 2 x 4096 taps at one rate: 32 KB per stream).
 *  - The first call creates the instance's FIR table.  Every stream's row starts from the words the stream runs with at that
 *    moment: the program's, or those of its set_param variant.  avdsp_b200_num_variants does not count the table.
 *  - The latest call wins for a word.  While a FIR table exists, set_param on tap words writes those streams' rows and creates
 *    no variant; set_param on any other word makes variants as before, and they combine with the rows.
 *  - reload_params drops the table.  reset keeps it: rows hold every fs column, so a reset to another rate runs that rate's taps.
 *  - Refusals change nothing: AVDSP_B200_ERR_UNSUPPORTED for a program without FIR taps, for DEVICE rows on a multi-device
 *    instance (HOST rows are split over its shards), and for a variant that changed a tap block's length; AVDSP_B200_ERR_ARG for
 *    a bad stream range, NULL values or an unknown memspace.
 *  - Kernels, DSP_FORMAT 2: the tensor-core FIR kernel runs per stream (bit-exact, as with shared taps); AUTO takes it for calls
 *    of at least 8192 frames, k_fir for shorter ones.  It keeps every stream's Toeplitz limb planes on the device, built from the
 *    rows before its first launch after they change: nStreams x paths x 4 x ((longest impulse rounded up to 128) / 128 + 1) x
 *    16 KB (C4, 2 x 4096 taps: 4.3 MB per stream, 4.4 GB for 1024 streams).  When they cannot be allocated the instance runs
 *    k_fir with its table (and says so in avdsp_b200_trace).  DSP_FORMAT 3: k_fir; AVDSP_B200_KERNEL_FIR_TC (the 3xTF32 form
 *    contracts with taps every stream shares) returns AVDSP_B200_ERR_UNSUPPORTED while a FIR table exists.
 *  - DSP_FORMAT 3: a row with a non-zero tap below 2^-60 (any fs column) sends its stream through the interpreter inside the same
 *    call, so every stream stays bit-exact (the FIR kernels' products could come near 2^-126, where they differ from the
 *    reference's multiply). */
int  avdsp_b200_set_fir_taps(avdsp_b200_t *, int firstStream, int nStreams, const int32_t *values, int memspace, void *cudaStream);

/* Per-stream state block, int32 words:  [0,dataSize) = the reference data area, same word offsets
 * (runtime/dsp_runtime.c:137-141);  then 8 aux words (xoshiro s0..s3, tpdfValue, tpdfRandom, current
 * global dither, pad -- the reference's process globals, runtime/dsp_tpdf.h:11-33);  then the 64-bit
 * LOAD_MEM/STORE_MEM words the reference keeps inside the code area (runtime/dsp_runtime.c:750-766). */
int  avdsp_b200_state_words(const avdsp_b200_t *);
int  avdsp_b200_data_size(const avdsp_b200_t *);
int  avdsp_b200_aux_offset(const avdsp_b200_t *);
int  avdsp_b200_mem_offset(const avdsp_b200_t *);
int  avdsp_b200_num_mem(const avdsp_b200_t *);
int  avdsp_b200_mem_word(const avdsp_b200_t *, int k);       /* code word index of MEM slot k */
int  avdsp_b200_get_state(avdsp_b200_t *, int stream, int32_t *words);
int  avdsp_b200_set_state(avdsp_b200_t *, int stream, const int32_t *words);

int  avdsp_b200_num_streams(const avdsp_b200_t *);
int  avdsp_b200_num_cores(const avdsp_b200_t *);
/* human-readable lowering trace (the counterpart of the reference's DSP_PRINTF>=2 opcode trace) */
const char *avdsp_b200_trace(const avdsp_b200_t *);
/* The same trace without an instance and without a CUDA device: validate + lower `prog` and plan the kernel geometries for
 * nStreams streams on a GPU with numSMs SMs (148 on B200); writes at most outLen-1 characters.  Returns totalLength or the
 * error codes of avdsp_b200_create.  Host-side inspection only: no kernel runs. */
int  avdsp_b200_describe(const int32_t *prog, int progWords, int fs, int format, int defaultDither, int nStreams, int numSMs,
                         char *out, int outLen);
/* message of the last failure in this thread ("" when none) */
const char *avdsp_b200_last_error(void);

/* Integer-pipe microbenchmark used for the INT roofline: runs `iters` dependent-free mad.wide.s32
 * per thread on the whole device and returns the achieved rate in mad.wide/s (0 on failure). */
double avdsp_b200_measure_int_peak(int device, int iters);
/* Float-pipe microbenchmark used for the FP32 roofline of the DSP_FORMAT 3 kernels: the reference's non-fused
 * multiply-accumulate (truncating multiply, runtime/dsp_ieee754.h:336-375, then a rounded add) as mul.rz.ftz.f32 +
 * add.rn.f32 (packed = 0) or mul.rz.ftz.f32x2 + add.rn.f32x2 (packed = 1); returns MACs per second. */
double avdsp_b200_measure_f32_peak(int device, int iters, int packed);

#ifdef __cplusplus
}
#endif
#endif /* AVDSP_B200_H_ */

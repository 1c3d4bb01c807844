/*
 * b200conv.h -- C ABI of the B200-native batched partitioned-FFT convolution engine.
 *
 * Drop-in boundary for ONE hot path of lsp-plugins/lsp-dsp-units: lsp::dspu::Convolver
 * (reference include/lsp-plug.in/dsp-units/util/Convolver.h:35-114,
 *  src/main/util/Convolver.cpp:36-340).  A "batch" is a set of independent convolver
 * instances (one mono-in / mono-out dspu::Convolver each) that live on one GPU and are
 * advanced together, one kernel sequence per audio block for all instances x partitions.
 * The C++ facade lsp::dspu::Convolver (lsp-dsp-units_b200/host) is a batch of one.
 *
 * Plain C: pointers and sizes only, no C++/torch types.  Every function returns
 * B200CONV_OK (0) or a negative error code; b200conv_last_error() gives the text.
 * There is no CPU fallback: without a CUDA device every call fails with
 * B200CONV_ERR_CUDA.
 */
#ifndef B200CONV_H_
#define B200CONV_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200CONV_RANK_MIN       8       /* CONVOLVER_RANK_MIN, Convolver.h:28 */
#define B200CONV_RANK_MAX       16      /* CONVOLVER_RANK_MAX, Convolver.h:29 */

enum
{
    B200CONV_OK             =  0,
    B200CONV_ERR_ARG        = -1,   /* bad argument (NULL handle, index out of range, rank mismatch) */
    B200CONV_ERR_NOMEM      = -2,   /* host or device allocation failed; previous state is intact     */
    B200CONV_ERR_CUDA       = -3,   /* CUDA runtime / launch failure, or no device                    */
    B200CONV_ERR_STATE      = -4    /* call not valid in the current state                            */
};

typedef struct b200conv_batch b200conv_batch_t;

/* Scheduler state of one instance; mirrors the observable part of Convolver.h:45-55. */
typedef struct b200conv_state
{
    size_t  conv_size;      /* nConvSize : taps given to init, 0 when not initialised (data_size()) */
    size_t  rank;           /* nRank     : clamped rank, 0 when not initialised (rank())            */
    size_t  frame_size;     /* nFrameSize: F = 2^(rank-1)                                            */
    size_t  frame_off;      /* nFrameOff : samples received in the current frame                    */
    size_t  bins;           /* ceil(conv_size / F) (Convolver.cpp:93)                                */
    size_t  partitions;     /* rows of IR spectra held on the device (bins + 1, folded overlap)      */
    size_t  part_offset;    /* first global partition index (partition-range sharding), else 0      */
    uint64_t frames;        /* complete frames received since init                                   */
} b200conv_state_t;

/* The 18 fields lsp::dspu::Convolver::dump writes (reference src/main/util/Convolver.cpp:315-337),
 * with the values the REFERENCE object would hold after the same init / process history:
 *   scalars   nDataBufferSize = (bins + 1) F (:137), nDirectSize = min(count, 128) (:141), nFrameSize,
 *             nFrameOff (:140, :298-311), nConvSize, nLevels (:165-181), nBlocks (:184-197),
 *             nBlocksDone (:198, :268-285: reset at a frame start, raised to
 *             min(nBlocks, size_t(nBlkInit + fBlkCoef * sub_id)) at every 128-sample boundary),
 *             nRank, nBlkInit, fBlkCoef (:199-210) -- all reproduced arithmetically (the engine itself
 *             has no raising levels and no load spreading);
 *   pointers  the reference reports slices of its host slab; the engine reports the DEVICE buffer
 *             that plays the same part: vDataBuffer -> pending block, vFrame -> frame in progress,
 *             vConvBuffer -> partial-spectrum scratch, vTaskData -> input-spectrum ring,
 *             vConvData -> folded IR spectra, vDirectData -> taps [0, F), vData -> the IR spectra
 *             allocation.  All NULL / 0 when the instance is not initialised (construct(), :46-69). */
typedef struct b200conv_dump
{
    const void *vDataBuffer, *vFrame, *vConvBuffer, *vTaskData, *vConvData, *vDirectData;
    size_t      nDataBufferSize, nDirectSize, nFrameSize, nFrameOff, nConvSize;
    size_t      nLevels, nBlocks, nBlocksDone, nRank, nBlkInit;
    float       fBlkCoef;
    const void *vData;
} b200conv_dump_t;

/* Counters since create (or the last b200conv_reset_stats). */
typedef struct b200conv_stats
{
    uint64_t launches;          /* kernels of this library launched                                 */
    uint64_t frames;            /* instance-frames pushed through the FFT -> MAC -> IFFT chain       */
    uint64_t h2d_bytes;         /* bytes copied host -> device by b200conv_process / _init          */
    uint64_t d2h_bytes;         /* bytes copied device -> host by b200conv_process                  */
    uint64_t mac_launches;      /* launches of the partition MAC kernel                             */
    uint64_t mac_algo_bytes;    /* algorithmic bytes of those launches (DESIGN.md: 16*F*bins + 24*F per instance-frame) */
    uint64_t mac_stream_bytes;  /* bytes those launches actually stream: less than mac_algo_bytes when one-frame calls
                                   run with lookahead (option "lookahead"), each IR spectrum row read once per K blocks */
} b200conv_stats_t;

/* ---- lifetime -------------------------------------------------------------------------- */

/* Creates a batch of `instances` un-initialised convolvers on CUDA device `device`
 * (-1 = the calling thread's current device).  Replaces N x Convolver::Convolver()
 * (Convolver.cpp:36-39). */
int     b200conv_create(b200conv_batch_t **out, int device, size_t instances);

/* Releases everything (N x Convolver::~Convolver, Convolver.cpp:41-44).  NULL is allowed. */
void    b200conv_free(b200conv_batch_t *h);

/* ---- Convolver::init / destroy --------------------------------------------------------- */

/* Convolver::init(data, count, rank, phase) for instance `idx` (Convolver.cpp:77-215):
 *   count == 0      -> the instance is destroyed and the call succeeds (:80-84);
 *   rank            -> clamped to [8, 16] (:87); all initialised instances of one batch must
 *                      share the clamped rank (B200CONV_ERR_ARG otherwise);
 *   phase           -> frame_off = size_t(phase * F) % F in fp32 (:140);
 *   `data` is a HOST pointer, borrowed for the call only.
 * The IR is transformed on the device.  All history of the instance is discarded (:110).
 * On allocation failure the previous state of the instance is kept (:103-108). */
int     b200conv_init(b200conv_batch_t *h, size_t idx, const float *data, size_t count,
                      size_t rank, float phase);

/* Same, for partition-range sharding of one long IR across GPUs: `data` holds the taps
 * [part_offset * F, part_offset * F + count) of the full IR and this instance produces only
 * their contribution; the full output is the sum over shards (SURVEY 8e).  part_offset == 0
 * is b200conv_init. */
int     b200conv_init_range(b200conv_batch_t *h, size_t idx, const float *data, size_t count,
                            size_t rank, float phase, size_t part_offset);

/* Convolver::init for `count` instances in ONE call (the IR ingest of a whole plugin / render job):
 * instance idx[k] gets data[k][0 .. counts[k]) with phases[k] (NULL: 0) and part_offsets[k] (NULL:
 * 0); counts[k] == 0 destroys it.  One device allocation, one staged asynchronous upload, one
 * transform launch over every partition of every instance.  Same rank rule, same failure
 * guarantee as b200conv_init (nothing changes unless everything was allocated). */
int     b200conv_init_many(b200conv_batch_t *h, size_t count, const size_t *idx, const float *const *data,
                           const size_t *counts, size_t rank, const float *phases,
                           const size_t *part_offsets);

/* Convolver::init for instance `idx` with the SAME impulse response and rank as the initialised
 * instance `src_idx` (many channels through one reverb): the device IR spectra are shared, only the
 * input-spectrum ring and the frame buffers are new.  The lender cannot be destroyed or
 * re-initialised while it is borrowed from (B200CONV_ERR_STATE). */
int     b200conv_init_shared(b200conv_batch_t *h, size_t idx, size_t src_idx, float phase);

/* Convolver::destroy for instance `idx` (Convolver.cpp:71-75); idempotent. */
int     b200conv_destroy(b200conv_batch_t *h, size_t idx);

/* ---- Convolver::process ---------------------------------------------------------------- */

/* N x Convolver::process(dst[i], src[i], count) (Convolver.cpp:217-313) in one call: HOST
 * pointers, one planar buffer of `count` floats per instance, any alignment, dst[i] == src[i]
 * allowed, any count (0 = no-op), state carried across calls, zero latency.  Instances that
 * are not initialised get zeros (:219-223).  Synchronous: dst is complete on return. */
int     b200conv_process(b200conv_batch_t *h, float *const *dst, const float *const *src,
                         size_t count);

/* Same for HOST buffers laid out as one planar matrix [instances][stride] floats (row i =
 * instance i): no per-instance pointer table, the rows go to the device with one strided copy
 * (a true DMA when the matrix is page-locked).  dst == src is allowed.  Synchronous. */
int     b200conv_process_planar(b200conv_batch_t *h, float *dst, const float *src,
                                size_t stride, size_t count);

/* Same with DEVICE buffers laid out [instances][stride] floats (row i = instance i), enqueued
 * on `stream` (a cudaStream_t; NULL = the batch's own stream) without host synchronisation.
 * dst == src is allowed.  All calls on one batch must be ordered on one stream (or be
 * separated by b200conv_sync). */
int     b200conv_process_device(b200conv_batch_t *h, float *dst, const float *src,
                                size_t stride, size_t count, void *stream);

/* Same with separate row strides for the two matrices. */
int     b200conv_process_device2(b200conv_batch_t *h, float *dst, size_t dst_stride,
                                 const float *src, size_t src_stride, size_t count, void *stream);

/* Waits for everything the batch has enqueued (own stream, and the latest call on a caller's stream).
 * Returns B200CONV_ERR_STATE if a bounded in-kernel wait has given up since the batch was created. */
int     b200conv_sync(b200conv_batch_t *h);

/* ---- partition-range sharding across GPUs: fused NVLink reduce ---------------------------- */

/* One long IR split by partition range over `world` GPUs (one process per GPU, each with a batch
 * of the same instances initialised through b200conv_init_range): instead of calling a
 * collective after every block, the launch tails exchange the partial output blocks over NVLink
 * peer memory themselves and rank 0 writes the SUMMED block to its dst (other ranks' dst is not
 * written).  Protocol:
 *   1. every rank: b200conv_reduce_prepare(h, grank, world, handle)  -> 64-byte CUDA IPC handle
 *      of its exchange buffer (call after the instances are initialised);
 *   2. exchange the handles between the processes (any transport; the tests use
 *      torch.distributed.all_gather), then every rank: b200conv_reduce_connect(h, all_handles);
 *   3. b200conv_process_device / _planar as usual, the same sequence of whole-frame calls on every
 *      rank (ranks 8..11; anything else returns B200CONV_ERR_STATE while connected);
 *   4. b200conv_reduce_disconnect(h).
 * b200conv_reduce_status reports whether any in-kernel wait for a peer timed out (2 s). */
#define B200CONV_IPC_HANDLE_BYTES   64
int     b200conv_reduce_prepare(b200conv_batch_t *h, int grank, int world, unsigned char *handle_out);
int     b200conv_reduce_connect(b200conv_batch_t *h, const unsigned char *all_handles);
int     b200conv_reduce_disconnect(b200conv_batch_t *h);
int     b200conv_reduce_status(b200conv_batch_t *h, int *timed_out);

/* ---- queries (Convolver.h:101,107) ------------------------------------------------------ */

size_t  b200conv_data_size(const b200conv_batch_t *h, size_t idx);
size_t  b200conv_rank(const b200conv_batch_t *h, size_t idx);
size_t  b200conv_instances(const b200conv_batch_t *h);
int     b200conv_get_state(const b200conv_batch_t *h, size_t idx, b200conv_state_t *st);
int     b200conv_get_dump(const b200conv_batch_t *h, size_t idx, b200conv_dump_t *out);
int     b200conv_get_stats(const b200conv_batch_t *h, b200conv_stats_t *st);
int     b200conv_reset_stats(b200conv_batch_t *h);

/* Per-launch timing of the partition MAC kernel (the roofline kernel): while enabled, every
 * k_mac launch is bracketed by CUDA events on the launching stream.  b200conv_get_profile
 * synchronises, returns the summed device time (ms) and launch count since the last call, and
 * clears the record.  Costs two event records per launch -- keep it off in timed regions. */
int     b200conv_set_profiling(b200conv_batch_t *h, int enable);
int     b200conv_get_profile(b200conv_batch_t *h, double *mac_ms, uint64_t *mac_launches);

/* The batch's own CUDA stream (cudaStream_t), for callers that time with CUDA events. */
void   *b200conv_stream(b200conv_batch_t *h);

/* Tuning / A-B knobs (value 0 = automatic unless stated):
 *   "mac_splits"  partition splits per instance-frame (1..32)
 *   "mac_stages"  shared-memory pipeline stages of the MAC stream (2..12)
 *   "fused"       1 (default) = ranks 8..13 run FFT + MAC + IFFT as ONE launch per block
 *                 (k_frame); 0 = always three launches (k_fwd, k_mac, k_inv)
 *   "fft_bias"    partitions taken off the split that also transforms the input (default 6)
 *   "pdl"         1 (default) = programmatic dependent launch between consecutive blocks
 *   "multi_frame" frames served by one pass over the IR spectra when a call brings several whole
 *                 frames: 8 (default), 4, 2, or 1 = off (one launch per frame)
 *   "eager"       1 (default) = after a synchronous host call has delivered block t, the partitions
 *                 q >= 1 of block t+1 are summed while the host is away; the next call then only
 *                 transforms its input, adds partition 0 and inverts (low call latency)
 *   "early_pend"  2 = that ahead-of-time sum starts while the launch that delivers block t is still
 *                 in its tail (back-to-back synchronous calls then run at the device rate);
 *                 0 = it starts after that launch has completed (lowest latency for a caller that
 *                 comes back once per audio block: nothing competes with the delivering launch);
 *                 1 (default) = automatic: early only while the caller keeps the GPU busy, i.e. the
 *                 previous ahead-of-time sum was still running when the call arrived
 *   "early_src"   when a one-launch-per-block kernel may transform its input block before every
 *                 earlier launch of the stream has completed (it may when no launch still in flight
 *                 writes that block; this takes the transform out of the launch-to-launch chain,
 *                 which matters for small batches): 0 = never; 1 (default) = on the batch's own
 *                 stream, where the library knows everything that is enqueued; 2 = on a caller's
 *                 stream too -- the caller promises that no kernel it enqueues between two calls
 *                 signals programmatic launch completion before it has written the input block
 *   "chain_ahead" ranks 14..16, whole-frame calls of one frame: 1 (default) = the partition sum of
 *                 block t + 1 (partitions q >= 1 need complete frames only) is launched behind the
 *                 inverse transform of block t and streams under it and under the transform of block
 *                 t + 1; partition 0 is added by that block's inverse transform.  Rows computed ahead
 *                 for a block that then arrives differently are simply not used; 0 = off
 *   "lookahead"   ranks 8..13, streams of one-frame calls in uniform mode: the launches of a group of
 *                 K blocks also sum, each over one bin slice, the partitions q >= 2K of the next
 *                 group's blocks (they need frames that are already in the ring), so each IR spectrum
 *                 row is streamed once per K blocks.  -1 (default) = automatic (bandwidth-bound
 *                 batches only); 0 = off; 2, 4, 8 = that K.  Results differ from "off" only in the
 *                 order of the partition sum
 *   "mac_tile"    developer knob, ranks 14..16, process-wide: bins per k_mac CTA (0 = 1024, 512, 256)
 *   "zero_copy"   1 (default) = b200conv_process_planar lets the kernels read / write page-locked
 *                 host matrices directly (no staging copies); 0 = always stage */
int     b200conv_set_option(b200conv_batch_t *h, const char *name, int value);

/* ---- the fastconv primitives on the device (lsp::dsp:: contract, SURVEY App. B) ---------- */

/* Batched device restatements of dsp::fastconv_parse / _apply / _parse_apply / _restore for
 * `count` independent problems at one rank (8..16).  All pointers are DEVICE pointers, rows are
 * contiguous.  An "image" here is 2^rank floats: 2^(rank-1) packed complex bins of the real
 * FFT, (DC, Nyquist) folded into bin 0 -- opaque to callers exactly like the reference's.
 *   parse       : image[i]  = FFT_{2^rank}([src[i][0 .. 2^(rank-1)), zeros])
 *   apply       : dst[i][0 .. 2^rank) += IFFT(c1[i] * c2[i]) / 2^rank
 *   parse_apply : dst[i][0 .. 2^rank) += IFFT(c[i] * parse(src[i])) / 2^rank
 *   restore     : dst[i][0 .. 2^rank)  = IFFT(image[i]) / 2^rank
 * Enqueued on `stream` (NULL = default stream of `device`) and truly stream-ordered: no host
 * synchronisation, no lock on the data path, no job upload (row i of every operand is problem i);
 * scratch comes from the stream-ordered allocator (cudaMallocAsync on `stream`). */
int     b200conv_fastconv_parse(int device, float *image, const float *src, size_t rank,
                                size_t count, void *stream);
int     b200conv_fastconv_apply(int device, float *dst, const float *c1, const float *c2,
                                size_t rank, size_t count, void *stream);
int     b200conv_fastconv_parse_apply(int device, float *dst, const float *c, const float *src,
                                      size_t rank, size_t count, void *stream);
int     b200conv_fastconv_restore(int device, float *dst, const float *image, size_t rank,
                                  size_t count, void *stream);

/* dsp::convolve (reference call site Convolver.cpp:295; same as the test helper
 * src/test/utest/util/convolver.cpp:32-40), batched on the device:
 *     dst[i][a + b] += src[i][a] * conv[i][b]    a < count, b < length
 * for `batch` independent problems; rows are `*_stride` floats apart (DEVICE pointers; dst rows hold
 * count + length - 1 valid samples and are accumulated into, like the reference's). */
int     b200conv_convolve(int device, float *dst, size_t dst_stride, const float *src, size_t src_stride,
                          const float *conv, size_t conv_stride, size_t length, size_t count,
                          size_t batch, void *stream);

/* ---- offline linear convolution ("next" row f1 of the scope table) -------------------------- */

/* Full linear convolution of `count` signals with ONE filter, host buffers:
 *     dst[i][0 .. nx + nh - 1) = src[i][0 .. nx) (*) h[0 .. nh)
 * The arithmetic core of SyncChirpProcessor::do_linear_convolution(s) without its padding / align
 * layout (that is b200conv_chirp_linear_convolutions below), run as ONE batched multi-frame pass of
 * the convolver engine: the filter is the impulse response (one set of spectra shared by all
 * signals), the signal zero-padded by nh - 1 is the input.
 * `rank` as in b200conv_init (partition = 2^(rank-1) samples); rows are `*_stride` floats apart.
 * Synchronous. */
int     b200conv_linear_convolve(int device, float *dst, size_t dst_stride, const float *src,
                                 size_t src_stride, size_t nx, size_t count, const float *h,
                                 size_t nh, size_t rank);

/* SyncChirpProcessor::do_linear_convolutions(Sample **data, size_t *offset, size_t nchannels,
 * size_t partSizeLimit) on plain arrays (reference src/main/util/SyncChirpProcessor.cpp:1374-1508):
 * every channel's recording, from its offset on, is convolved with the processor's inverse filter
 * in partitions of nPartitionSize samples.
 *
 *   b200conv_chirp_plan   calculateConvolutionPartitionSize (:1224-1250) and
 *                         calculateConvolutionParameters (:1299-1331): partition size = the power of
 *                         two >= min(part_size_limit, 32768) (0 means 32768), rank = log2 + 1; per
 *                         channel vPartitions = max(in_len, inverse_len) / partition + 1,
 *                         vPaddedLengths, vInversePrepends, vConvLengths = 2 * padded, vAlignOffsets;
 *                         allocation_size = the largest vConvLengths = samples per result channel.
 *                         The per-channel arrays (nchannels entries each) may be NULL.
 *   b200conv_chirp_linear_convolutions
 *                         inputs[ch] = data[ch]->channel(0, offset[ch]) (HOST), in_len[ch] =
 *                         data[ch]->length() - offset[ch]; result = pConvResult, [nchannels] rows of
 *                         result_stride >= allocation_size floats (HOST), zeroed here and then filled
 *                         like the reference's: the convolution of the tail-padded input with the
 *                         PREPEND-padded inverse filter lands at vAlignOffsets[ch] (:1499), and the
 *                         first vConvLengths[ch] samples of the row are multiplied by `scale`
 *                         (= fConvScale / fs^2; dsp::mul_k2 at :1508 starts at index 0).  Null
 *                         partitions (:1457-1460, :1476-1479) contribute nothing either way.
 *                         Runs as ONE batched multi-frame pass of the convolver engine; channels of
 *                         equal padded length share one set of filter spectra.  Partition sizes
 *                         below 128 (rank < 8) are not supported (B200CONV_ERR_ARG).  Synchronous. */
typedef struct b200conv_chirp_plan
{
    size_t  partition_size;     /* sConvParams.nPartitionSize */
    size_t  conv_rank;          /* sConvParams.nConvRank      */
    size_t  image;              /* sConvParams.nImage (the reference's image size, informative) */
    size_t  allocation_size;    /* sConvParams.nAllocationSize */
} b200conv_chirp_plan_t;

int     b200conv_chirp_plan(b200conv_chirp_plan_t *plan, size_t *partitions, size_t *padded,
                            size_t *prepends, size_t *conv_lengths, size_t *align_offsets,
                            const size_t *in_len, size_t nchannels, size_t inverse_len,
                            size_t part_size_limit);
int     b200conv_chirp_linear_convolutions(int device, float *result, size_t result_stride,
                                           const float *const *inputs, const size_t *in_len,
                                           size_t nchannels, const float *inverse, size_t inverse_len,
                                           size_t part_size_limit, float scale);

/* ---- Equalizer, FIR / FFT modes ("next" row f2 of the scope table) --------------------------- */

/* The DATA PATH of lsp::dspu::Equalizer in its EQM_FIR / EQM_FFT modes for a batch of equalizers:
 * one-partition overlap-add convolution with nFirSize = 2^fir_rank samples of latency and a
 * cross-fade when a kernel is handed over smoothly.  The filter DESIGN (FilterBank,
 * Filter::freq_chart, window) stays with the caller: the boundary is the point where the
 * reference calls dsp::fastconv_parse on the finished impulse response.
 *
 *   b200conv_eq_create        buffers of Equalizer::init(filters, fir_rank)
 *                             (reference src/main/filters/Equalizer.cpp:96-121); fir_rank in [7, 15]
 *   b200conv_eq_set_kernel    Equalizer::reconfigure's hand-over (Equalizer.cpp:336-345): `ir` holds
 *                             nFirSize taps (host); smooth = 0 replaces the kernel at once (vConv),
 *                             smooth != 0 installs it as vNewConv and raises EF_XFADE, consumed by
 *                             the next block boundary (:486-501)
 *   b200conv_eq_clear         EF_CLEAR (Equalizer.cpp:273-278), all instances
 *   b200conv_eq_process*      Equalizer::process, EQM_FIR / EQM_FFT case (Equalizer.cpp:474-518),
 *                             for ALL instances in one call: host pointer per instance, one planar
 *                             host matrix, or device matrices (stream-ordered, never synchronises;
 *                             stream NULL = the batch's own stream)
 *   b200conv_eq_latency       the data path's share of Equalizer::get_latency(): nFirSize (the
 *                             other nFirSize / 2 of Equalizer.cpp:347 is the kernel's own delay)
 */
typedef struct b200conv_eq b200conv_eq_t;

int     b200conv_eq_create(b200conv_eq_t **out, int device, size_t instances, size_t fir_rank);
void    b200conv_eq_free(b200conv_eq_t *e);
int     b200conv_eq_set_kernel(b200conv_eq_t *e, size_t idx, const float *ir, int smooth);
int     b200conv_eq_clear(b200conv_eq_t *e);
int     b200conv_eq_process(b200conv_eq_t *e, float *const *dst, const float *const *src, size_t samples);
int     b200conv_eq_process_planar(b200conv_eq_t *e, float *dst, const float *src, size_t stride,
                                   size_t samples);
int     b200conv_eq_process_device(b200conv_eq_t *e, float *dst, size_t dst_stride, const float *src,
                                   size_t src_stride, size_t samples, void *stream);
int     b200conv_eq_sync(b200conv_eq_t *e);
void   *b200conv_eq_stream(b200conv_eq_t *e);
size_t  b200conv_eq_fir_size(const b200conv_eq_t *e);
size_t  b200conv_eq_latency(const b200conv_eq_t *e);
size_t  b200conv_eq_instances(const b200conv_eq_t *e);

/* ---- SpectralProcessor ("next" row f4 of the scope table) ------------------------------------ */

/* lsp::dspu::SpectralProcessor for a batch of instances (reference
 * include/lsp-plug.in/dsp-units/util/SpectralProcessor.h, src/main/util/SpectralProcessor.cpp): an
 * STFT with a sine window before and after the spectral operation, frames of N = 2^rank samples
 * every N / 2, N samples of latency.  ONE launch per process call for all instances, whatever
 * their phases and the call size.
 *
 *   b200conv_sp_create        N x SpectralProcessor::init(max_rank) (:58-75); ranks 7..15
 *   b200conv_sp_set_rank      set_rank (:133-141) for the whole batch (one launch shape): ignored
 *                             when equal to the current rank or above max_rank; drops history and
 *                             every bound table (tables are rank-specific: bind again)
 *   b200conv_sp_set_phase     set_phase (:127-131), per instance, clamped to [0, 1]; takes effect at
 *                             the next process call like the reference's update_settings (:107-125):
 *                             buffers cleared, first transform after N/2 - size_t(N * (phase / 2)) samples
 *   b200conv_sp_bind_complex  the reference binds a HOST callback that edits the packed complex
 *   b200conv_sp_bind_gain     spectrum (spectral_processor_func_t, SpectralProcessor.h:38); on the
 *   b200conv_sp_unbind        device the spectral operation is a per-instance table instead:
 *                             spectrum[k] *= H[k] (`table`: 2^rank packed complex bins, host) or
 *                             spectrum[k] *= g[k] (`gain`: 2^rank real values, host).  Any table is
 *                             allowed -- the result is Re(IFFT(X H)) exactly as the reference's with
 *                             that callback.  Unbound (:174-175): the frames are only windowed.
 *   b200conv_sp_process_*     SpectralProcessor::process(dst, src, count) (:143-199) for all
 *                             instances: device matrices [instances][stride] (stream-ordered, dst ==
 *                             src allowed) or one planar host matrix (synchronous)
 *   b200conv_sp_reset         reset() (:247-257);  b200conv_sp_remaining  remaining() (:241-245);
 *   b200conv_sp_latency       latency() = 2^rank */
typedef struct b200conv_sp b200conv_sp_t;

int     b200conv_sp_create(b200conv_sp_t **out, int device, size_t instances, size_t max_rank);
void    b200conv_sp_free(b200conv_sp_t *s);
int     b200conv_sp_set_rank(b200conv_sp_t *s, size_t rank);
int     b200conv_sp_set_phase(b200conv_sp_t *s, size_t idx, float phase);
int     b200conv_sp_bind_complex(b200conv_sp_t *s, size_t idx, const float *table);
int     b200conv_sp_bind_gain(b200conv_sp_t *s, size_t idx, const float *gain);
int     b200conv_sp_unbind(b200conv_sp_t *s, size_t idx);
int     b200conv_sp_process_device(b200conv_sp_t *s, float *dst, size_t dst_stride, const float *src,
                                   size_t src_stride, size_t count, void *stream);
int     b200conv_sp_process_planar(b200conv_sp_t *s, float *dst, const float *src, size_t stride, size_t count);
int     b200conv_sp_reset(b200conv_sp_t *s);
int     b200conv_sp_sync(b200conv_sp_t *s);
void   *b200conv_sp_stream(b200conv_sp_t *s);
size_t  b200conv_sp_rank(const b200conv_sp_t *s);
size_t  b200conv_sp_latency(const b200conv_sp_t *s);
size_t  b200conv_sp_remaining(const b200conv_sp_t *s, size_t idx);
size_t  b200conv_sp_instances(const b200conv_sp_t *s);

/* ---- scope-table row f4, second sibling: lsp::dspu::SpectralSplitter, batched --------------------
 * Reference: src/main/util/SpectralSplitter.cpp (+ include/lsp-plug.in/dsp-units/util/SpectralSplitter.h).
 * One forward transform of the last 2^rank input samples every 2^(chunk_rank - 1) samples, shared by
 * all bound handlers ("bands"); each band applies its function to the spectrum, transforms back,
 * windows with sin^2 and overlap-adds into its own output stream (latency 2^chunk_rank).
 * lsp::dspu::FFTCrossover is this class with a real gain curve per band (FFTCrossover.cpp:124-140).
 *   b200conv_ss_create          N x SpectralSplitter::init(max_rank, handlers) (:64-130); ranks 7..14
 *   b200conv_ss_set_rank        set_rank (:271-278), for the whole batch; ignored when equal or above
 *                               the maximum; the bound tables are rank-specific: bind again afterwards
 *   b200conv_ss_set_chunk_rank  set_chunk_rank (:280-287): <= 0 = the transform rank, else clamped to [5, rank]
 *   b200conv_ss_set_phase       set_phase (:264-268), per instance, clamped to [0, 1]; like every setter
 *                               it takes effect at the next process call, which clears that instance's
 *                               buffers (update_settings, :227-245)
 *   b200conv_ss_bind_complex    the reference binds HOST callbacks per handler: a function on the packed
 *   b200conv_ss_bind_gain       complex spectrum (spectral_splitter_func_t, SpectralSplitter.h:44) and a
 *   b200conv_ss_bind_sink       sink for the processed samples (spectral_splitter_sink_t, :60).  On the
 *   b200conv_ss_unbind(_all)    device the function is a per-(instance, handler) table -- 2^rank packed
 *                               complex bins, or 2^rank real gains (FFTCrossover's band) -- or absent
 *                               (bind_sink: the input frames themselves, :327), and the sink of handler h
 *                               is row h of the output.  bind clears the handler's output buffer (:175-176);
 *                               unbind of an unbound handler fails (STATUS_NOT_BOUND, :190-191)
 *   b200conv_ss_process_*       SpectralSplitter::process(src, count) (:296-383) for all instances in ONE
 *                               launch: dst[h * band_stride + instance * dst_stride + i]; rows of handlers
 *                               that are not bound are left untouched; an instance with nothing bound does
 *                               nothing at all (:301-302)
 *   b200conv_ss_clear           clear() (:247-260);  b200conv_ss_latency  latency() = 2^chunk_rank (:289-296) */
typedef struct b200conv_ss b200conv_ss_t;

int     b200conv_ss_create(b200conv_ss_t **out, int device, size_t instances, size_t max_rank, size_t handlers);
void    b200conv_ss_free(b200conv_ss_t *s);
int     b200conv_ss_set_rank(b200conv_ss_t *s, size_t rank);
int     b200conv_ss_set_chunk_rank(b200conv_ss_t *s, long rank);
int     b200conv_ss_set_phase(b200conv_ss_t *s, size_t idx, float phase);
int     b200conv_ss_bind_complex(b200conv_ss_t *s, size_t idx, size_t handler, const float *table);
int     b200conv_ss_bind_gain(b200conv_ss_t *s, size_t idx, size_t handler, const float *gain);
int     b200conv_ss_bind_sink(b200conv_ss_t *s, size_t idx, size_t handler);
int     b200conv_ss_unbind(b200conv_ss_t *s, size_t idx, size_t handler);
int     b200conv_ss_unbind_all(b200conv_ss_t *s, size_t idx);
size_t  b200conv_ss_bindings(const b200conv_ss_t *s, size_t idx);
int     b200conv_ss_process_device(b200conv_ss_t *s, float *dst, size_t band_stride, size_t dst_stride,
                                   const float *src, size_t src_stride, size_t count, void *stream);
int     b200conv_ss_process_planar(b200conv_ss_t *s, float *dst, const float *src, size_t stride, size_t count);
int     b200conv_ss_clear(b200conv_ss_t *s);
int     b200conv_ss_sync(b200conv_ss_t *s);
void   *b200conv_ss_stream(b200conv_ss_t *s);
size_t  b200conv_ss_rank(const b200conv_ss_t *s);
size_t  b200conv_ss_chunk_rank(const b200conv_ss_t *s);
size_t  b200conv_ss_latency(const b200conv_ss_t *s);
size_t  b200conv_ss_instances(const b200conv_ss_t *s);
size_t  b200conv_ss_handlers(const b200conv_ss_t *s);

/* ---- matrix convolver: many inputs x many outputs through routed impulse responses ----------
 * `inputs` I and `outputs` O at one rank, and a list of routes (input i, output o, impulse response h).
 * Every call produces, with zero latency, for every output
 *     y_o[n] = sum over the routes r with output(r) = o of  sum_k h_r[k] x_input(r)[n - k]
 * over every sample since the last b200conv_mx_set_routes / b200conv_mx_clear.  The arithmetic plan is
 * the convolver's (uniform partitions of F = 2^(rank-1) samples, folded overlap, a frequency-domain
 * delay line); what is shared is ONE input-spectrum ring per input, whatever the number of routes that
 * read it, and ONE inverse transform per output, whatever the number of routes summed into it.  A
 * true-stereo reverb (2 x 2, 4 routes), an ambisonic room response (1 x 16) or a binaural decoder
 * (16 x 2, each ear a sum of 16 convolutions) is one object.
 *
 *   b200conv_mx_create          ranks 8..16 (B200CONV_ERR_ARG otherwise), 1..4096 inputs and outputs;
 *                               until the first set_routes every output is zeros
 *   b200conv_mx_set_routes      replaces the whole routing: route r reads input[r], adds into output[r]
 *                               through ir[r][0 .. length[r]) (HOST pointers, borrowed for the call only).
 *                               length[r] >= 1, indices in range, each (input, output) pair at most once,
 *                               else B200CONV_ERR_ARG; count == 0 is valid (every output is zeros).  All
 *                               input history is discarded.  On B200CONV_ERR_ARG / _ERR_NOMEM nothing
 *                               changes (the old routes and history stay).  Ordered after every call
 *                               already enqueued on the object; synchronous
 *   b200conv_mx_set_irs         replaces the IRs of some routes and KEEPS the input history: route
 *                               route[k] (its index in the last set_routes) gets ir[k][0 .. length[k])
 *                               (HOST pointers, copied to page-locked staging before the call returns).
 *                               With k counting samples from the first sample of the next process call
 *                               and w(k) = min(1, (k + 1) / fade) (w = 1 when fade == 0: a hard switch),
 *                               a changed route contributes (1 - w) h_old (*) x + w h_new (*) x, both
 *                               over the whole history since set_routes / clear; once the fade is over
 *                               the new IRs stay.  B200CONV_ERR_ARG: route out of range or twice, NULL
 *                               or empty IR, or an IR of more partitions than the ring reaches
 *                               (ceil(length / F) + 1 > the longest route's at set_routes: use
 *                               set_routes); B200CONV_ERR_STATE: a fade is in progress.  On any error
 *                               nothing changes; count == 0 is a no-op; a one-tap zero IR fades a route
 *                               out.  Enqueued on `stream` (NULL = the object's own) like
 *                               process_device, with stream-ordered allocations; the host waits only
 *                               while the previous call's staging is still being uploaded.  During a
 *                               fade each launch group runs the delta routes (G_new - G_old) into
 *                               extra outputs and one blend launch.  clear ends a fade with the new
 *                               IRs in place; set_routes discards it
 *   b200conv_mx_fade_remaining  samples of the fade not yet covered by the calls enqueued so far
 *                               (0: no fade); host arithmetic, never waits
 *   b200conv_mx_clear           discards the input history, keeps the routes
 *   b200conv_mx_process_device  src: DEVICE matrix [inputs][src_stride], dst: DEVICE matrix
 *                               [outputs][dst_stride] floats; count must be a multiple of F (0 = no-op;
 *                               anything else returns B200CONV_ERR_ARG and changes nothing).  Outputs with
 *                               no route get zeros; dst == src with equal strides is allowed.  Enqueued on
 *                               `stream` (a cudaStream_t; NULL = the object's own stream) without host
 *                               synchronisation; all calls on one object must be ordered on one stream (or
 *                               be separated by b200conv_mx_sync)
 *   b200conv_mx_process_planar  the same on HOST matrices; synchronous
 *   b200conv_mx_sync            waits for everything the object has enqueued
 *   b200conv_mx_frame_size      F: the call-size granule
 *   b200conv_mx_routes          routes of the current routing */
typedef struct b200conv_mx b200conv_mx_t;

int     b200conv_mx_create(b200conv_mx_t **out, int device, size_t inputs, size_t outputs, size_t rank);
void    b200conv_mx_free(b200conv_mx_t *m);
int     b200conv_mx_set_routes(b200conv_mx_t *m, size_t count, const size_t *input, const size_t *output,
                               const float *const *ir, const size_t *length);
int     b200conv_mx_set_irs(b200conv_mx_t *m, size_t count, const size_t *route,
                            const float *const *ir, const size_t *length, size_t fade, void *stream);
size_t  b200conv_mx_fade_remaining(const b200conv_mx_t *m);
int     b200conv_mx_clear(b200conv_mx_t *m);
int     b200conv_mx_process_device(b200conv_mx_t *m, float *dst, size_t dst_stride, const float *src,
                                   size_t src_stride, size_t count, void *stream);
int     b200conv_mx_process_planar(b200conv_mx_t *m, float *dst, size_t dst_stride, const float *src,
                                   size_t src_stride, size_t count);
int     b200conv_mx_sync(b200conv_mx_t *m);
void   *b200conv_mx_stream(b200conv_mx_t *m);
size_t  b200conv_mx_inputs(const b200conv_mx_t *m);
size_t  b200conv_mx_outputs(const b200conv_mx_t *m);
size_t  b200conv_mx_rank(const b200conv_mx_t *m);
size_t  b200conv_mx_frame_size(const b200conv_mx_t *m);
size_t  b200conv_mx_routes(const b200conv_mx_t *m);

/* ---- misc -------------------------------------------------------------------------------- */

const char *b200conv_last_error(void);      /* thread-local text of the last failure */
const char *b200conv_version(void);

#ifdef __cplusplus
}
#endif

#endif /* B200CONV_H_ */

/*
 * kernels.cuh -- sm_100a device code of the batched partitioned-FFT convolver.
 *
 * Kernel map (reference primitive it replaces -> kernel):
 *   dsp::fastconv_parse  (Convolver.cpp:159,174,191,270)  -> k_fwd   : F reals -> M packed bins
 *   dsp::fastconv_apply  (Convolver.cpp:280-285, the hot   -> k_mac   : sum_q G_q * X_{t-q}
 *        loop: nBlocks x (spectrum multiply + IFFT + add)     k_inv   : ONE inverse FFT per frame
 *   the three above for one audio block, all instances     -> k_frame : one launch per block
 *        x partitions (ranks 8..13), blocks overlapped        (+ fused NVLink reduce of
 *        on the device                                         partition-range shards)
 *   ... for several frames of one call                     -> k_mac_multi : one pass over the IR
 *                                                             spectra serves up to 8 frames
 *   dsp::fastconv_parse_apply head (Convolver.cpp:256,293) -> folded into partition q = 0
 *   dsp::convolve        (Convolver.cpp:295)               -> k_partial (unaligned call sizes),
 *                                                             k_convolve (exported primitive)
 *   dsp::copy/move/fill_zero (Convolver.cpp:291,296,308-310) -> ring indices, nothing moves
 *
 * Notation: rank R, N = 2^R, F = M = N/2 (frame length = packed complex bins), P = M/2.
 *
 * Spectrum layout: M float2 per row; bin k = 1..M-1 complex, bin 0 = (DC, Nyquist), both real.
 */
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <type_traits>

namespace b200conv
{

/* ------------------------------------------------------------------------------------------- */
/* Descriptors shared with the host                                                             */

struct InstDesc                     /* one per instance, device resident */
{
    const float2   *G;              /* [nq][M]   folded IR spectra, row q_local = q - q_lo          */
    float2         *ring;           /* [S][M]    input-spectrum ring; frame t lives in slot (-t) mod S */
    float          *cur;            /* [F]       frame being received (partial-call path)           */
    float          *pend;           /* [F]       contribution of complete frames to that frame      */
    const float    *head;           /* [F]       taps [0, F) in the time domain                     */
    int64_t         t_delta;        /* frames(instance) - frames(batch), uniform mode               */
    uint32_t        nq;             /* rows in G                                                    */
    uint32_t        q_lo;           /* global index of row 0                                        */
    uint32_t        S;              /* ring slots                                                   */
    uint32_t        pad;
};

struct Job                          /* explicit work item (general path, init, primitives) */
{
    const float    *src;            /* transform input: F samples (caller's block, or the instance's `cur`) */
    float          *dst;            /* inverse-transform output: F samples (caller's block, or `pend`)      */
    float2         *spec;           /* ring row that receives the spectrum                                  */
    const float    *psrc;           /* P1: n samples of the call -> cur[off ..), answered from the OLD pend  */
    float          *pdst;
    const float    *psrc2;          /* P2: n2 samples of the call -> cur[off2 ..), answered from the NEW pend */
    float          *pdst2;
    uint32_t        inst;
    uint32_t        slot0;          /* ring slot of X_t for this job's frame index t                */
    uint32_t        qa, qb;         /* global partition range of the MAC                            */
    uint32_t        off, n;         /* P1: first sample index in the frame, sample count            */
    uint32_t        off2, n2;       /* P2                                                           */
    uint32_t        tlo;            /* low 32 bits of the job's frame index t                       */
    uint32_t        flags;          /* JOB_*                                                        */
};

/* What one job of the general (any call size, any phase) path asks of its k_frame launch, in this
 * order:  P1 (samples that continue the frame in progress)  ->  FFT (the frame is complete: its
 * spectrum enters the ring)  ->  MAC over [qa, qb) + inverse transform into dst  ->  P2 (the first
 * samples of the next frame, answered from the block just computed). */
enum { JOB_FFT = 1, JOB_MAC = 2,
       JOB_FFT_PREV = 4 /* the transformed frame is t - 1 (the MAC prepares frame t): publish t, not t + 1 */ };

/* A short job list travels in the kernel's parameter space (constant bank: no copy operation in
 * the stream, no trip across PCIe or to DRAM before a CTA knows what to do) -- the latency of a
 * real-time call is one kernel launch.  Longer lists are uploaded to device memory (StepArgs::jobs). */
constexpr uint32_t JOB_PACK = 16;
struct JobPack
{
    Job j[JOB_PACK];
};

struct StepArgs                     /* by-value kernel argument */
{
    const InstDesc *inst;
    const Job      *jobs;           /* NULL -> uniform mode: jobs are derived from the fields below */
    const uint32_t *active;         /* uniform mode: instance ids                                   */
    const float2   *tw;             /* N-point twiddle table exp(-2 pi i j / N)                     */
    float2         *ypart;          /* [job][split][M] partial spectra                              */
    float          *park;           /* k_inv_half: [job][2][F] half results (odd, even); NULL = not available */
    uint32_t       *ring_head;      /* [instance] frames whose spectrum is in the ring (low 32 bits) */
    uint32_t       *error;          /* host-mapped word: set when a bounded in-kernel wait gave up    */
    uint32_t       *slot_done;      /* k_frame: [FRAME_SLOTS][n_cap] sequence number + 1 of the launch whose tail
                                       last finished with that (slot, instance); NULL: launches are not pipelined */
    uint32_t        seq;            /* k_frame: sequence number of this launch (its slot is seq % FRAME_SLOTS) */
    uint32_t        n_cap;          /* k_frame: instances of the batch (row pitch of slot_done)        */
    uint32_t        rows;           /* partial rows per job in ypart (0 = splits); a launch writes rows
                                       row0 .. row0 + splits - 1, the inverse transform sums all `rows` */
    uint32_t        row0;
    uint32_t        sum0;           /* k_frame: the inverse transform sums rows sum0 .. rows - 1 (the pending
                                       MAC has folded its rows into row sum0 = row0 - 1: fold_tickets)      */
    uint32_t       *chain_head;     /* k_mac in the three-kernel block (ranks 14..16), != NULL: one word per batch,
                                       "the spectra of all frames < *chain_head are final".  The launch of block t
                                       polls it for t before its first read of the ring (its own CTAs may be
                                       running while the transforms of EARLIER blocks are still resident: every
                                       kernel of the chain releases its successor at its top) and publishes
                                       t + 1 once the transform of block t has completed. */
    uint32_t       *fold_tickets;   /* k_mac: [job] counters (zero between launches); != NULL: the last CTA of a job
                                       adds the job's rows row0 .. row0 + splits - 1, in order, into the last one */
    const float    *src;            /* uniform mode: [instances][stride]                            */
    float          *dst;
    uint64_t        stride;         /* uniform mode: floats between instance rows of src            */
    uint64_t        stride_dst;     /* ... of dst                                                   */
    uint64_t        t_base;         /* uniform mode: batch frame counter of frame 0 of this launch  */
    uint32_t        n_active;
    uint32_t        n_jobs;
    uint32_t        splits;
    uint32_t        rank;
    uint32_t        frame0;         /* uniform mode: first frame (within the call) of this launch   */
    uint32_t        flags;
    /* k_frame lookahead (one-frame-per-call streams, see LA_BUFS): la_K = 0 -> off */
    float2         *la_T;           /* [LA_BUFS][n_jobs][la_K][splits][M] tail sums T of a group's blocks    */
    uint32_t       *la_prod;        /* [LA_BUFS][n_cap] CTAs that have written their tail rows into that buffer */
    uint32_t       *la_cons;        /* [LA_BUFS][n_cap] launch tails that have read their T rows from it     */
    uint32_t        la_K;           /* group size K (2, 4, 8)                                               */
    uint32_t        la_c;           /* this launch's block within its group: it streams bin slice la_c      */
    uint32_t        la_use;         /* T of this block is complete: the launch sums partitions q < 2K only  */
    uint32_t        la_put, la_get; /* buffer this launch writes (next group) / reads (its own group)       */
    uint32_t        la_put_need;    /* la_cons[la_put] must reach this before the first tail-row write      */
    uint32_t        la_get_need;    /* la_prod[la_get] must reach this before the T rows are read           */
};

enum { INV_FULL = 1, STEP_FROM_Q1 = 2, STEP_HEAD_ONLY = 4,
       STEP_AFTER_FWD = 128 /* k_mac launched with programmatic serialisation right behind the k_fwd of the
                               SAME block (three-kernel path, ranks 14..16): the CTAs of split 0 take the
                               stage that needs the arriving frame's spectrum last, after griddepcontrol.wait */,
       STEP_LINEAR_JOBS = 64 /* IR ingest / the fastconv primitives: forward job j transforms src + j * F into
                                the spectrum row (float2 *) dst + j * F; inverse job j writes dst + j * stride_dst */,
       STEP_HOST_IO = 8 /* src / dst are page-locked HOST matrices: no bulk-copy staging */,
       STEP_WAIT_HEAD = 16 /* k_mac launched early (programmatic serialization) behind a k_frame:
                              poll ring_head before touching the newest spectra */,
       STEP_ORDER_DST = 256 /* k_frame: the output block overlaps a block that a launch which may still be in
                               flight writes or reads (a buffer re-used every call, a cascade's hand-over
                               block): this launch keeps the full griddepcontrol.wait before its first
                               shared write, i.e. its tail starts after every earlier launch has completed */,
       STEP_AHEAD = 512 /* k_mac of the three-kernel block (ranks 14..16), launched one block AHEAD (behind the
                           inverse transform of block t - 1, with STEP_FROM_Q1): partitions q >= 1 of block t need
                           complete frames only, so it streams under that inverse transform and under the transform
                           of block t.  Its rows go to a slot of their own (no wait in front of the row write), what
                           it reads is ordered by chain_head, and only CTA (0, 0) waits for the launches before it,
                           as its last instruction (completion order) */,
       STEP_Q0_IN_INV = 1024 /* k_inv / k_inv_half: add partition 0 -- G_0 times the block's own spectrum -- while
                                summing the partial rows (the MAC ran ahead, STEP_AHEAD), and publish chain_head */,
       STEP_EARLY_SRC = 32 /* k_frame: the input block may be read before griddepcontrol.wait -- set by
                              the host only when the predecessor on the stream is this batch's own pending
                              k_mac and the input is a caller-owned HOST block no kernel writes */ };

/* Partition-range sharding across GPUs (one long IR, SURVEY 8e): every rank's k_frame produces a
 * PARTIAL output block; the sum is formed inside the launch tails over NVLink peer memory --
 * no collective library call, no host in the loop, no root: an ALL-TO-ALL exchange after which
 * every rank holds the summed block (added in rank order, hence bit-identical on all ranks).
 *   every rank g : the CTA that finishes channel c of block b inverse-transforms its partial
 *                  spectrum and stores the block into slot [b % depth][g][c] of EVERY peer's exchange
 *                  buffer as 8-byte words { sample bits, sequence number b + 1 } (posted peer stores;
 *                  an 8-byte store is never torn, so a word whose sequence number matches carries
 *                  its sample: no fence, no separate flag, one NVLink crossing of latency);
 *                  then polls its own slots [b % depth][p][c] word by word until the sequence numbers
 *                  read b + 1, adds the world blocks, writes the output block, and tells every rank
 *                  that it has consumed block b of channel c (the slot is reused by block b + depth).
 * Sequence numbers, not resettable counters: a late peer can never be mistaken for the next
 * block.  All waits are bounded (a peer that never shows up raises *error instead of hanging the
 * GPU; the host then fails the next call). */
/* k_frame launches of one batch are pipelined FRAME_SLOTS deep: launch s keeps its partial rows, its
 * tickets (and, sharded, its own output block) in slot s % FRAME_SLOTS, so the tail of block t --
 * sum of the partial rows, inverse transform, cross-GPU exchange -- overlaps the partition stream
 * AND the tail of block t + 1 instead of gating it.  What orders the launches:
 *   slot reuse     slot_done[slot][instance] holds s + 1 once the tail of launch s (the previous user
 *                  of the slot is launch s - FRAME_SLOTS) has finished; CTAs of launch s poll for
 *                  s + 1 - FRAME_SLOTS before their first write into the slot (bounded; in steady
 *                  state it is long there);
 *   output blocks  a launch whose output block overlaps a block that a launch in flight writes or reads
 *                  (the host's launch history sees it: STEP_ORDER_DST) keeps the full
 *                  griddepcontrol.wait before its first shared write;
 *   completion     the tail CTAs execute griddepcontrol.wait as their LAST instruction, so launch
 *                  s completes after launch s - 1 (stream order for whatever follows). */
constexpr int FRAME_SLOTS      = 4;
/* Lookahead for streams of one-frame calls (k_frame, la_K = K > 0).  Blocks are grouped K at a time
 * (group g = blocks t0 .. t0 + K - 1).  y_t needs  head_t = sum_{q < 2K} G_q X_{t-q}  and the tail
 * T_t = sum_{q >= 2K} G_q X_{t-q}, which reads frames <= t - 2K only.  For every block of group g + 1
 * that is a frame <= t0 - 1, so the K launches of group g compute the tails of group g + 1, launch
 * t0 + c the bin slice [c M / K, (c + 1) M / K) of all K of them: each IR spectrum row is streamed
 * once per group instead of once per block.  A launch sums its own head (or, when the tails of its
 * group are not complete -- the first group after any interruption -- every partition), adds the
 * split rows of its T (written by the K launches before it), and inverts.  Every T value has one
 * writer and the summation order is fixed: results do not depend on timing or on the overlap.
 * Ordering (all waits bounded, per instance, sequence counts the host predicts):
 *   T complete   la_prod[buf] counts producer CTAs (st.release after the rows); the tail CTA of a
 *                consumer polls it before reading its T rows (launch t0 + K reads rows that launch
 *                t0 + K - 1 may still be writing);
 *   T reuse      LA_BUFS = 3 buffers rotate by group; la_cons[buf] counts the consumers that have
 *                read their rows; a producer polls it before its first row write (the last reader
 *                of a buffer is K + 1 launches before its next writer, so it is long done there). */
constexpr int LA_BUFS          = 3;
constexpr int REDUCE_MAX_WORLD = 8;
constexpr int REDUCE_DEPTH     = 4;
struct ReduceArgs
{
    uint32_t    mode;                               /* 0 = off */
    uint32_t    world, grank;
    uint32_t    t0;                                 /* frame counter (low 32 bits) at connect time */
    uint32_t    channels;                           /* instances per rank */
    uint32_t    frame;                              /* F */
    uint2      *words[REDUCE_MAX_WORLD];            /* rank p's [depth][world][channels][F] {bits, seq}  (p == grank: local) */
    uint32_t   *consumed[REDUCE_MAX_WORLD];         /* rank p's [world][channels]: blocks rank g has consumed, written by g */
    float      *scratch;                            /* local [channels][F]: this rank's own block */
};

__device__ __forceinline__ uint64_t global_ns()
{
    uint64_t t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

#ifdef B200CONV_TIMING
/* developer instrumentation (tools/frame_timeline.py, gen_timeline.py, chain_timeline.py): per-CTA timestamps of the last k_frame launch */
__device__ unsigned long long g_frame_times[8192 * 8];
#define FRAME_STAMP(slot)   do { if ((threadIdx.x == 0) && (blockIdx.x < 8192)) g_frame_times[blockIdx.x * 8 + (slot)] = global_ns(); } while (0)
#define CHAIN_STAMP(id, slot) do { if ((threadIdx.x == 0) && ((id) < 8192)) g_frame_times[(id) * 8 + (slot)] = global_ns(); } while (0)
#else
#define FRAME_STAMP(slot)   do { } while (0)
#define CHAIN_STAMP(id, slot) do { } while (0)
#endif

__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t *p)
{
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

__device__ __forceinline__ uint32_t ld_acquire_gpu(const uint32_t *p)
{
    uint32_t v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

/* Bounded in-kernel waits.  Every spin in this file has a deadline: a predecessor that faulted
 * (or a peer GPU that never shows up) must not hang the device.  A waiter that gives up stores a
 * code into *err -- a host-mapped word the host checks at its next synchronisation point, which
 * then fails with B200CONV_ERR_STATE -- and carries on (its output is garbage, the GPU is alive). */
constexpr uint64_t SPIN_LIMIT_NS = 2000000000ull;
enum { SPIN_ERR_RING = 1, SPIN_ERR_PEER = 2 };

__device__ __forceinline__ void spin_fail(uint32_t *err, uint32_t code)
{
    if (err != nullptr)
        *reinterpret_cast<volatile uint32_t *>(err) = code;
}

/* waits until int32(*p - need) >= 0; SYS: the word is written by another GPU */
template <bool SYS>
__device__ __forceinline__ void wait_ge(const uint32_t *p, uint32_t need, uint32_t *err, uint32_t code)
{
    uint32_t have   = SYS ? ld_acquire_sys(p) : ld_acquire_gpu(p);
    if (int32_t(have - need) >= 0)
        return;
    const uint64_t deadline = global_ns() + SPIN_LIMIT_NS;
    for (uint32_t n = 1; ; ++n)
    {
        __nanosleep(SYS ? 200 : 100);
        have            = SYS ? ld_acquire_sys(p) : ld_acquire_gpu(p);
        if (int32_t(have - need) >= 0)
            return;
        if (((n & 31u) == 0) && (global_ns() > deadline))
        {
            spin_fail(err, code);
            return;
        }
    }
}

__device__ __forceinline__ uint32_t rows_per_job(const StepArgs &a)
{
    return (a.rows != 0) ? a.rows : a.splits;
}

__device__ __forceinline__ Job fetch_job(const StepArgs &a, uint32_t j)
{
    if (a.jobs != nullptr)
        return a.jobs[j];
    if (a.flags & STEP_LINEAR_JOBS)
    {
        const uint64_t F    = 1ull << (a.rank - 1);
        Job r;
        r.src               = a.src + uint64_t(j) * F;
        r.spec              = reinterpret_cast<float2 *>(a.dst) + uint64_t(j) * F;
        r.dst               = a.dst + uint64_t(j) * a.stride_dst;       /* inverse transforms: output row */
        r.psrc = r.psrc2    = nullptr;
        r.pdst = r.pdst2    = nullptr;
        r.inst = r.slot0 = r.qa = r.qb = r.off = r.n = r.off2 = r.n2 = r.tlo = r.flags = 0;
        return r;
    }

    /* uniform mode: every active instance sits on a frame boundary and receives whole frames */
    const uint32_t F    = 1u << (a.rank - 1);
    uint32_t ia         = j % a.n_active;
    uint32_t f          = a.frame0 + j / a.n_active;
    Job r;
    r.inst              = a.active[ia];
    const InstDesc &d   = a.inst[r.inst];
    uint64_t t          = uint64_t(int64_t(a.t_base) + d.t_delta) + f;
    uint32_t tm         = uint32_t(t % d.S);
    r.slot0             = (tm == 0) ? 0 : d.S - tm;
    r.tlo               = uint32_t(t);
    r.flags             = JOB_FFT | JOB_MAC;
    r.psrc = r.psrc2    = nullptr;
    r.pdst = r.pdst2    = nullptr;
    r.off2 = r.n2       = 0;
    r.src               = a.src + uint64_t(r.inst) * a.stride + uint64_t(f) * F;
    r.dst               = a.dst + uint64_t(r.inst) * a.stride_dst + uint64_t(f) * F;
    r.spec              = d.ring + uint64_t(r.slot0) * F;
    r.qa                = d.q_lo;
    r.qb                = d.q_lo + d.nq;
    if (a.flags & STEP_FROM_Q1)         /* complete frames only: what is pending for the frame about to arrive */
        r.qa                = max(r.qa, 1u);
    if (a.flags & STEP_HEAD_ONLY)       /* the arriving frame's own partition; the rest is already in ypart */
        r.qb                = min(r.qb, 1u);
    r.off               = 0;
    r.n                 = 0;
    return r;
}

/* ------------------------------------------------------------------------------------------- */
/* Small complex helpers                                                                        */

__device__ __forceinline__ float2 cadd(float2 a, float2 b)  { return make_float2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ float2 csub(float2 a, float2 b)  { return make_float2(a.x - b.x, a.y - b.y); }
__device__ __forceinline__ float2 cconj(float2 a)           { return make_float2(a.x, -a.y); }
__device__ __forceinline__ float2 cmul(float2 a, float2 b)
{
    return make_float2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x);
}
/* L2-coherent 16-byte load; volatile so that a group of them stays in program order (all issued
 * before the first use) instead of being sunk next to their consumers */
__device__ __forceinline__ float4 ld_cg_f4(const float4 *p)
{
    float4 v;
    asm volatile("ld.global.cg.v4.f32 {%0, %1, %2, %3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p) : "memory");
    return v;
}

/* a * conj(b) */
__device__ __forceinline__ float2 cmulc(float2 a, float2 b)
{
    return make_float2(a.x * b.x + a.y * b.y, a.y * b.x - a.x * b.y);
}

/* ------------------------------------------------------------------------------------------- */
/* Shared-memory Stockham FFT: NH independent P-point transforms laid out back to back.         */
/* Radix 4, with one leading radix-2 pass when log2(P) is odd.  Every pass stages its inputs in  */
/* registers.  With a second buffer (PP) a pass is load A -> butterflies -> store B -> barrier;  */
/* without it, load -> barrier -> store -> barrier in place.                                    */

template <int RANK, int TT = 0, int NHO = 0>    /* TT: threads doing the transform (0 = natural count); NHO: override of NH */
struct FftCfg
{
    static constexpr int N      = 1 << RANK;
    static constexpr int M      = N / 2;
    static constexpr int P      = M / 2;
    static constexpr int LOGP   = RANK - 2;
    static constexpr int NH     = (NHO > 0) ? NHO : (RANK >= 16) ? 1 : 2;  /* halves resident in smem */
    static constexpr int BF     = NH * P / 4;                           /* radix-4 butterflies/pass */
    static constexpr int T      = (TT > 0) ? TT : ((BF >= 512) ? 512 : ((BF < 32) ? 32 : BF));
    static constexpr int BPT    = (BF + T - 1) / T;                     /* butterflies per thread   */
    static constexpr bool PP    = (RANK <= 12);                         /* ping-pong work buffers   */
    static constexpr bool TWS   = (RANK <= 12);                         /* twiddle table in smem    */
    static constexpr int WORK   = NH * P;                               /* float2 per work buffer   */

    /* Twiddle table layout (float2 entries; built by make_twiddles on the host).  Every access a
     * warp makes is unit-stride in its lane index, so the shared-memory copy is conflict-free:
     *   [0, TW_PRE)            radix-4 passes in execution order (Ns = NS0, 4 NS0, ... < P), each
     *                          3 * Ns entries: exp(-2 pi i k r / (4 Ns)), r = 1, 2, 3, k < Ns
     *   [TW_PRE, TW_POST)      w_M^m = exp(-2 pi i m / M), m < P       (odd-half pre/post twiddle)
     *   [TW_POST, TW_TOTAL)    w_N^k = exp(-2 pi i k / N), k <= M/2    (real-FFT split / merge)     */
    static constexpr int NS0    = (LOGP & 1) ? 2 : 1;
    static constexpr int TW_PRE = P - NS0;                              /* 3 * (NS0 + 4 NS0 + ... + P/4) */
    static constexpr int TW_POST = TW_PRE + P;
    static constexpr int TW_TOTAL = TW_POST + M / 2 + 1;
    /* Ranks >= 13 have no room for the whole table next to the work buffer, but the passes need only
     * ONE factor per butterfly (w^2, w^3 by multiplication): a compact copy of the r = 1 third of
     * every pass, (P - NS0) / 3 entries (44 KiB at rank 16), keeps the dependent twiddle loads of
     * every pass on chip instead of in L2. */
    static constexpr int TWC_N  = (P - NS0) / 3;
    static constexpr size_t SMEM = (size_t(WORK) * (PP ? 2 : 1) + (TWS ? TW_TOTAL : TWC_N)) * sizeof(float2);
};

/* Transforms the NH sequences held in A; returns the buffer that holds the result (A or B). */
/* WMUL: one twiddle load per butterfly, w^2 and w^3 by multiplication (a few 1e-8 of error).
 * Always on where the table is read from global memory / L2 (ranks >= 12); throughput-bound
 * callers turn it on for the shared-memory table too, where it saves two of three LDS. */
/* FAST1: the first, twiddle-free pass (stride 1) is a radix-8 pass when log2(P) is odd (it
 * replaces the radix-2 pass and the first radix-4 pass) and a radix-4 pass otherwise, and its
 * outputs -- 64 / 32 contiguous bytes per thread -- leave as 16-byte stores whose order is
 * rotated per lane so that every quarter-warp covers all 32 banks.  (The plain passes store
 * 8 bytes at a 16 .. 64 byte lane stride: 2- to 4-way bank conflicts, the largest share of the
 * shared-memory wavefronts of a throughput-bound caller.) */
template <bool INV>
__device__ __forceinline__ float2 rot90(float2 z)       /* forward: -i z ; inverse: +i z */
{
    return INV ? make_float2(-z.y, z.x) : make_float2(z.y, -z.x);
}

/* TWC: `tw` is the compact table (see FftCfg::TWC_N): pass Ns at offset (Ns - NS0) / 3, r = 1 only. */
template <int RANK, bool INV, bool PP, int TT = 0, bool WMUL = (RANK >= 12), bool FAST1 = true, int NHO = 0,
          bool TWC = false>
__device__ __forceinline__ float2 *fft_smem(float2 *A, float2 *B, const float2 *tw, int tid)
{
    static_assert((!TWC) || WMUL, "fft_smem: the compact table holds one factor per butterfly");
    using C = FftCfg<RANK, TT, NHO>;
    constexpr int P = C::P, T = C::T, BPT = C::BPT, NH = C::NH;

    constexpr bool USE16 = (!PP) && WMUL && FAST1 && (BPT >= 4) && ((NH * P / 16) % T == 0);
    float2 *in  = A;
    float2 *out = PP ? B : A;
    int Ns = 1;
    if constexpr (FAST1 && USE16 && !(C::LOGP & 1))
    {
        /* radix-16, Ns = 1: no twiddles, outputs 16 j .. 16 j + 15 are contiguous (128 bytes per thread):
         * eight 16-byte stores whose order is rotated per lane, so that the eight lanes of every
         * quarter-warp cover all 32 banks */
        constexpr int IT16  = USE16 ? (NH * P / 16) / T : 1;
        float2 v[IT16][16];
        #pragma unroll
        for (int i = 0; i < IT16; ++i)
        {
            int idx = tid + i * T;
            int h   = idx / (P / 16), j = idx % (P / 16);
            #pragma unroll
            for (int r = 0; r < 16; ++r)
                v[i][r] = in[h * P + j + r * (P / 16)];
        }
        __syncthreads();
        const int sw = tid & 7;
        #pragma unroll
        for (int i = 0; i < IT16; ++i)
        {
            int idx = tid + i * T;
            int h   = idx / (P / 16), j = idx % (P / 16);
            float2 (&x)[16] = v[i];
            auto dft4 = [](float2 &a, float2 &b, float2 &c, float2 &d)
            {
                float2 s0 = cadd(a, c), s1 = csub(a, c), s2 = cadd(b, d), s3 = rot90<INV>(csub(b, d));
                a = cadd(s0, s2); b = cadd(s1, s3); c = csub(s0, s2); d = csub(s1, s3);
            };
            #pragma unroll
            for (int s2 = 0; s2 < 4; ++s2)
                dft4(x[s2], x[4 + s2], x[8 + s2], x[12 + s2]);
            {
                const float c1 = 0.92387953251128674f, s1 = 0.38268343236508977f, r2 = 0.70710678118654752f;
                auto cw = [&](float2 &z, float wr, float wi)
                {
                    z = INV ? make_float2(z.x * wr - z.y * wi, z.y * wr + z.x * wi)
                            : make_float2(z.x * wr + z.y * wi, z.y * wr - z.x * wi);
                };
                cw(x[4 * 1 + 1], c1, s1);   cw(x[4 * 1 + 2], r2, r2);   cw(x[4 * 1 + 3], s1, c1);
                cw(x[4 * 2 + 1], r2, r2);   x[4 * 2 + 2] = rot90<INV>(x[4 * 2 + 2]);   cw(x[4 * 2 + 3], -r2, r2);
                cw(x[4 * 3 + 1], s1, c1);   cw(x[4 * 3 + 2], -r2, r2);  cw(x[4 * 3 + 3], -c1, -s1);
            }
            #pragma unroll
            for (int r1 = 0; r1 < 4; ++r1)
                dft4(x[4 * r1], x[4 * r1 + 1], x[4 * r1 + 2], x[4 * r1 + 3]);
            /* output r = r1 + 4 r2 sits in x[4 r1 + r2]; chunk c = outputs 2 c, 2 c + 1 */
            float4 c[8];
            #pragma unroll
            for (int n = 0; n < 8; ++n)
            {
                const int ra = 2 * n, rb = 2 * n + 1;
                const float2 a = x[4 * (ra & 3) + (ra >> 2)], b = x[4 * (rb & 3) + (rb >> 2)];
                c[n]    = make_float4(a.x, a.y, b.x, b.y);
            }
            /* e_n = chunk (n + sw) & 7, by a three-stage barrel rotation */
            float4 d[8], e[8], f[8];
            #pragma unroll
            for (int n = 0; n < 8; ++n)
                d[n]    = (sw & 1) ? c[(n + 1) & 7] : c[n];
            #pragma unroll
            for (int n = 0; n < 8; ++n)
                e[n]    = (sw & 2) ? d[(n + 2) & 7] : d[n];
            #pragma unroll
            for (int n = 0; n < 8; ++n)
                f[n]    = (sw & 4) ? e[(n + 4) & 7] : e[n];
            float4 *row = reinterpret_cast<float4 *>(out + h * P + 16 * j);
            #pragma unroll
            for (int n = 0; n < 8; ++n)
                row[(n + sw) & 7]   = f[n];
        }
        __syncthreads();
        Ns = 16;
    }
    else if (FAST1 && (C::LOGP & 1))
    {
        constexpr int B8    = NH * P / 8;                       /* radix-8 butterflies */
        constexpr int IT8   = (B8 + T - 1) / T;
        float2 v[IT8][8];
        #pragma unroll
        for (int i = 0; i < IT8; ++i)
        {
            int idx = tid + i * T;
            if (idx < B8)
            {
                int h   = idx / (P / 8), j = idx % (P / 8);
                #pragma unroll
                for (int r = 0; r < 8; ++r)
                    v[i][r] = in[h * P + j + r * (P / 8)];
            }
        }
        if (!PP)
            __syncthreads();
        const int sw = (tid >> 1) & 3;                          /* per-lane rotation of the four 16-byte chunks */
        #pragma unroll
        for (int i = 0; i < IT8; ++i)
        {
            int idx = tid + i * T;
            if (idx < B8)
            {
                int h   = idx / (P / 8), j = idx % (P / 8);
                const float r2 = 0.70710678118654752f;
                float2 a0 = cadd(v[i][0], v[i][4]), a1 = csub(v[i][0], v[i][4]);
                float2 a2 = cadd(v[i][2], v[i][6]), a3 = rot90<INV>(csub(v[i][2], v[i][6]));
                float2 a4 = cadd(v[i][1], v[i][5]), a5 = csub(v[i][1], v[i][5]);
                float2 a6 = cadd(v[i][3], v[i][7]), a7 = rot90<INV>(csub(v[i][3], v[i][7]));
                float2 b0 = cadd(a0, a2), b2 = csub(a0, a2), b1 = cadd(a1, a3), b3 = csub(a1, a3);
                float2 b4 = cadd(a4, a6), b6 = rot90<INV>(csub(a4, a6));
                float2 t5 = cadd(a5, a7), t7 = csub(a5, a7);
                /* w8 = (1 -+ i) / sqrt 2 ; w8^3 = (-1 -+ i) / sqrt 2  (forward / inverse) */
                float2 b5 = INV ? make_float2((t5.x - t5.y) * r2, (t5.x + t5.y) * r2)
                                : make_float2((t5.x + t5.y) * r2, (t5.y - t5.x) * r2);
                float2 b7 = INV ? make_float2((-t7.x - t7.y) * r2, (t7.x - t7.y) * r2)
                                : make_float2((t7.y - t7.x) * r2, (-t7.x - t7.y) * r2);
                float2 V0 = cadd(b0, b4), V1 = cadd(b1, b5), V2 = cadd(b2, b6), V3 = cadd(b3, b7);
                float2 V4 = csub(b0, b4), V5 = csub(b1, b5), V6 = csub(b2, b6), V7 = csub(b3, b7);
                float4 c0 = make_float4(V0.x, V0.y, V1.x, V1.y), c1 = make_float4(V2.x, V2.y, V3.x, V3.y);
                float4 c2 = make_float4(V4.x, V4.y, V5.x, V5.y), c3 = make_float4(V6.x, V6.y, V7.x, V7.y);
                /* e_n = chunk (n + sw) & 3, by a two-stage barrel rotation */
                float4 d0 = (sw & 1) ? c1 : c0, d1 = (sw & 1) ? c2 : c1, d2 = (sw & 1) ? c3 : c2, d3 = (sw & 1) ? c0 : c3;
                float4 e0 = (sw & 2) ? d2 : d0, e1 = (sw & 2) ? d3 : d1, e2 = (sw & 2) ? d0 : d2, e3 = (sw & 2) ? d1 : d3;
                float4 *row = reinterpret_cast<float4 *>(out + h * P + 8 * j);
                row[(0 + sw) & 3]   = e0;
                row[(1 + sw) & 3]   = e1;
                row[(2 + sw) & 3]   = e2;
                row[(3 + sw) & 3]   = e3;
            }
        }
        __syncthreads();
        if (PP) { float2 *t = in; in = out; out = t; }
        Ns = 8;
    }
    else if (FAST1)
    {
        /* radix-4, Ns = 1: no twiddles, outputs 4 j .. 4 j + 3 are contiguous */
        float2 v[BPT][4];
        #pragma unroll
        for (int i = 0; i < BPT; ++i)
        {
            int idx = tid + i * T;
            if (idx < NH * P / 4)
            {
                int h   = idx / (P / 4), j = idx % (P / 4);
                #pragma unroll
                for (int r = 0; r < 4; ++r)
                    v[i][r] = in[h * P + j + r * (P / 4)];
            }
        }
        if (!PP)
            __syncthreads();
        const int sw = (tid >> 2) & 1;
        #pragma unroll
        for (int i = 0; i < BPT; ++i)
        {
            int idx = tid + i * T;
            if (idx < NH * P / 4)
            {
                int h   = idx / (P / 4), j = idx % (P / 4);
                float2 s0 = cadd(v[i][0], v[i][2]), s1 = csub(v[i][0], v[i][2]);
                float2 s2 = cadd(v[i][1], v[i][3]), rot = rot90<INV>(csub(v[i][1], v[i][3]));
                float2 V0 = cadd(s0, s2), V1 = cadd(s1, rot), V2 = csub(s0, s2), V3 = csub(s1, rot);
                float4 c0 = make_float4(V0.x, V0.y, V1.x, V1.y), c1 = make_float4(V2.x, V2.y, V3.x, V3.y);
                float4 *row = reinterpret_cast<float4 *>(out + h * P + 4 * j);
                row[sw]     = sw ? c1 : c0;
                row[sw ^ 1] = sw ? c0 : c1;
            }
        }
        __syncthreads();
        if (PP) { float2 *t = in; in = out; out = t; }
        Ns = 4;
    }
    else if (C::LOGP & 1)
    {
        /* radix-2, Ns = 1: twiddles are all 1.  NH*P/2 butterflies = 2*BPT per thread. */
        float2 a[2 * BPT], b[2 * BPT];
        #pragma unroll
        for (int i = 0; i < 2 * BPT; ++i)
        {
            int idx = tid + i * T;
            if (idx < NH * P / 2)
            {
                int h   = idx / (P / 2), j = idx % (P / 2);
                a[i]    = in[h * P + j];
                b[i]    = in[h * P + j + P / 2];
            }
        }
        if (!PP)
            __syncthreads();
        #pragma unroll
        for (int i = 0; i < 2 * BPT; ++i)
        {
            int idx = tid + i * T;
            if (idx < NH * P / 2)
            {
                int h   = idx / (P / 2), j = idx % (P / 2);
                out[h * P + 2 * j]      = cadd(a[i], b[i]);
                out[h * P + 2 * j + 1]  = csub(a[i], b[i]);
            }
        }
        __syncthreads();
        if (PP) { float2 *t = in; in = out; out = t; }
        Ns = 2;
    }

    /* Radix-16 passes (two radix-4 layers fused in registers) where a thread owns at least 16 points
     * per pass and the transform runs in place (ranks 14..16): the passes of these ranks are bound by
     * shared-memory round trips and barriers, and there are half as many this way.  Leading radix-4
     * passes bring Ns to >= 16 (their stores have the bank rotation below) and the remaining factor
     * to a power of 16. */
    auto pass16 = [&](int Ns)
    {
        constexpr int IT16  = USE16 ? (NH * P / 16) / T : 1;
        float2 v[IT16][16];
        #pragma unroll
        for (int i = 0; i < IT16; ++i)
        {
            int idx = tid + i * T;
            int h   = idx / (P / 16), j = idx % (P / 16);
            #pragma unroll
            for (int r = 0; r < 16; ++r)
                v[i][r] = in[h * P + j + r * (P / 16)];
        }
        __syncthreads();
        /* exp(-2 pi i k / (16 Ns)) is the r = 1 entry of the radix-4 pass 4 Ns, its fourth power that of pass Ns */
        const float2 *t1 = tw + (TWC ? (4 * Ns - C::NS0) / 3 : (4 * Ns - C::NS0));
        const float2 *t4 = tw + (TWC ? (Ns - C::NS0) / 3 : (Ns - C::NS0));
        #pragma unroll
        for (int i = 0; i < IT16; ++i)
        {
            int idx = tid + i * T;
            int h   = idx / (P / 16), j = idx % (P / 16);
            int k   = j & (Ns - 1);
            float2 (&x)[16] = v[i];
            {
                const float2 w1 = t1[k], w4 = t4[k];
                const float2 w2 = cmul(w1, w1), w3 = cmul(w2, w1), w8 = cmul(w4, w4), w12 = cmul(w8, w4);
                auto tw_mul = [&](float2 &z, float2 w) { z = INV ? cmulc(z, w) : cmul(z, w); };
                tw_mul(x[1], w1);   tw_mul(x[2], w2);   tw_mul(x[3], w3);   tw_mul(x[4], w4);
                tw_mul(x[5], cmul(w4, w1));  tw_mul(x[6], cmul(w4, w2));  tw_mul(x[7], cmul(w4, w3));
                tw_mul(x[8], w8);
                tw_mul(x[9], cmul(w8, w1));  tw_mul(x[10], cmul(w8, w2)); tw_mul(x[11], cmul(w8, w3));
                tw_mul(x[12], w12);
                tw_mul(x[13], cmul(w12, w1)); tw_mul(x[14], cmul(w12, w2)); tw_mul(x[15], cmul(w12, w3));
            }
            auto dft4 = [](float2 &a, float2 &b, float2 &c, float2 &d)
            {
                float2 s0 = cadd(a, c), s1 = csub(a, c), s2 = cadd(b, d), s3 = rot90<INV>(csub(b, d));
                a = cadd(s0, s2); b = cadd(s1, s3); c = csub(s0, s2); d = csub(s1, s3);
            };
            /* layer A: over s1 of x[4 s1 + s2]; result y[s2][r1] lands in x[4 r1 + s2] */
            #pragma unroll
            for (int s2 = 0; s2 < 4; ++s2)
                dft4(x[s2], x[4 + s2], x[8 + s2], x[12 + s2]);
            /* y[s2][r1] *= w16^(s2 r1) */
            {
                const float c1 = 0.92387953251128674f, s1 = 0.38268343236508977f, r2 = 0.70710678118654752f;
                auto cw = [&](float2 &z, float wr, float wi)     /* times (wr - i wi) forward, (wr + i wi) inverse */
                {
                    z = INV ? make_float2(z.x * wr - z.y * wi, z.y * wr + z.x * wi)
                            : make_float2(z.x * wr + z.y * wi, z.y * wr - z.x * wi);
                };
                cw(x[4 * 1 + 1], c1, s1);   cw(x[4 * 1 + 2], r2, r2);   cw(x[4 * 1 + 3], s1, c1);
                cw(x[4 * 2 + 1], r2, r2);   x[4 * 2 + 2] = rot90<INV>(x[4 * 2 + 2]);   cw(x[4 * 2 + 3], -r2, r2);
                cw(x[4 * 3 + 1], s1, c1);   cw(x[4 * 3 + 2], -r2, r2);  cw(x[4 * 3 + 3], -c1, -s1);
            }
            /* layer B: over s2 of x[4 r1 + s2]; X[r1 + 4 r2] lands in x[4 r1 + r2] */
            #pragma unroll
            for (int r1 = 0; r1 < 4; ++r1)
                dft4(x[4 * r1], x[4 * r1 + 1], x[4 * r1 + 2], x[4 * r1 + 3]);
            float2 *o  = out + h * P + ((j - k) << 4) + k;
            #pragma unroll
            for (int r1 = 0; r1 < 4; ++r1)
                #pragma unroll
                for (int r2 = 0; r2 < 4; ++r2)
                    o[(r1 + 4 * r2) * Ns]   = x[4 * r1 + r2];
        }
        __syncthreads();
    };

    auto pass4 = [&](int Ns)
    {
        float2 v[BPT][4];
        #pragma unroll
        for (int i = 0; i < BPT; ++i)
        {
            int idx = tid + i * T;
            if (idx < NH * P / 4)
            {
                int h   = idx / (P / 4), j = idx % (P / 4);
                #pragma unroll
                for (int r = 0; r < 4; ++r)
                    v[i][r] = in[h * P + j + r * (P / 4)];
            }
        }
        if (!PP)
            __syncthreads();

        const float2 *tws = tw + (TWC ? (Ns - C::NS0) / 3 : (Ns - C::NS0));    /* this pass: 3 * Ns entries, r-major (see FftCfg) */
        #pragma unroll
        for (int i = 0; i < BPT; ++i)
        {
            int idx = tid + i * T;
            if (idx < NH * P / 4)
            {
                int h   = idx / (P / 4), j = idx % (P / 4);
                int k   = j & (Ns - 1);
                float2 x0 = v[i][0], x1 = v[i][1], x2 = v[i][2], x3 = v[i][3];
                if (Ns > 1)
                {
                    float2 w1 = tws[k];
                    float2 w2 = WMUL ? cmul(w1, w1) : tws[Ns + k];
                    float2 w3 = WMUL ? cmul(w2, w1) : tws[2 * Ns + k];
                    if (INV)    { x1 = cmulc(x1, w1); x2 = cmulc(x2, w2); x3 = cmulc(x3, w3); }
                    else        { x1 = cmul(x1, w1);  x2 = cmul(x2, w2);  x3 = cmul(x3, w3);  }
                }
                float2 s0 = cadd(x0, x2), s1 = csub(x0, x2);
                float2 s2 = cadd(x1, x3), s3 = csub(x1, x3);
                /* forward: rot = -i * s3 ; inverse: rot = +i * s3 */
                float2 rot = INV ? make_float2(-s3.y, s3.x) : make_float2(s3.y, -s3.x);
                float2 *o  = out + h * P + ((j - k) << 2) + k;
                float2 V0 = cadd(s0, s2), V1 = cadd(s1, rot), V2 = csub(s0, s2), V3 = csub(s1, rot);
                if (FAST1 && (Ns < 16))
                {
                    /* Strides 4 and 8: a half-warp holds 4 / 2 groups of Ns consecutive lanes whose
                     * outputs for one r fall into the same banks.  Group g stores its outputs in the
                     * order r = g, g+1, ... instead (a barrel rotation of four registers), which
                     * spreads the groups over all 32 banks. */
                    const int rn = (Ns == 4) ? ((tid >> 2) & 3) : ((tid >> 3) & 1);
                    float2 d0 = (rn & 1) ? V1 : V0, d1 = (rn & 1) ? V2 : V1, d2 = (rn & 1) ? V3 : V2, d3 = (rn & 1) ? V0 : V3;
                    float2 e0 = (rn & 2) ? d2 : d0, e1 = (rn & 2) ? d3 : d1, e2 = (rn & 2) ? d0 : d2, e3 = (rn & 2) ? d1 : d3;
                    o[((0 + rn) & 3) * Ns]  = e0;
                    o[((1 + rn) & 3) * Ns]  = e1;
                    o[((2 + rn) & 3) * Ns]  = e2;
                    o[((3 + rn) & 3) * Ns]  = e3;
                }
                else
                {
                    o[0]        = V0;
                    o[Ns]       = V1;
                    o[2 * Ns]   = V2;
                    o[3 * Ns]   = V3;
                }
            }
        }
        __syncthreads();
        if (PP) { float2 *t = in; in = out; out = t; }
    };

    if constexpr (USE16)
    {
        /* remaining factor P / Ns = 4^m: radix-4 until Ns >= 16 and m is even, then radix-16 */
        #pragma unroll 1
        while ((Ns < 16) || (((31 - __clz(P / Ns)) & 3) != 0))
        {
            pass4(Ns);
            Ns <<= 2;
        }
        #pragma unroll 1
        for ( ; Ns < P; Ns <<= 4)
            pass16(Ns);
    }
    else
    {
        for ( ; Ns < P; Ns <<= 2)
            pass4(Ns);
    }
    return in;
}

/* ------------------------------------------------------------------------------------------- */
/* fwd_body : F real samples (zero padded to 2F) -> M packed complex bins.                       */
/*                                                                                             */
/* z[m] = x[2m] + i x[2m+1], m < P (the upper half of the packed sequence is the zero padding).  */
/* Even bins of its M-point transform are FFT_P(z), odd bins are FFT_P(z * w_M^m); the real-FFT  */
/* split then needs Z[k] and Z[M-k], which have the same parity, so the two halves never mix.    */
/* twg = twiddle table in global memory (used next to the global loads), tw = the table the      */
/* transform passes read (shared-memory copy when the caller staged one, else twg).              */

template <int RANK, bool PP, int TT = 0, bool SMEM_OUT = false, bool WM = (RANK >= 12), int NHO = 0, bool TWC = false>
__device__ __forceinline__ void fwd_body(float2 *A, float2 *B, const float *src, float2 *out,
                                         const float2 *twg, const float2 *tw, int tid,
                                         float2 **smem_out = nullptr, int only_pass = -1)
{
    /* TWC: `tw` is the compact pass table (fft_smem); every other lookup goes to twg */
    const float2 *twx       = TWC ? twg : tw;
    /* only_pass (one resident half, NH == 1): 0 = even bins only, 1 = odd bins only -- the two
     * halves of a frame are independent all the way to the output row (k_fwd_half) */
    /* SMEM_OUT (ping-pong ranks only): the bins go to whichever work buffer the transform did
     * not end in, reported through *smem_out; `out` is ignored */
    static_assert((!SMEM_OUT) || (PP && (FftCfg<RANK, TT, NHO>::NH == 2)), "fwd_body: SMEM_OUT needs two work buffers");
    using C = FftCfg<RANK, TT, NHO>;
    constexpr int P = C::P, M = C::M, T = C::T, NH = C::NH;

    #pragma unroll 1
    for (int pass = 0; pass < 2 / NH; ++pass)
    {
        if ((only_pass >= 0) && (pass != only_pass))
            continue;
        /* The streaming phases (this load and the split pass below) run at one CTA per SM on the big
         * ranks: their global loads are issued LB at a time before the first use, or each thread
         * would sit out a full memory latency per element (profiles/: 60 % of the rank-16 transform
         * was long-scoreboard stall in these two loops). */
        static_assert(P % T == 0, "fwd_body: whole rounds");
        constexpr int LB = (P / T >= 8) ? 8 : (P / T);
        const bool src8 = (reinterpret_cast<uintptr_t>(src) & 7) == 0;
        const bool need_w = (NH == 2) || (pass == 1);
        #pragma unroll 1
        for (int m0 = tid; m0 < P; m0 += LB * T)
        {
            float2 z[LB], w[LB];
            #pragma unroll
            for (int u = 0; u < LB; ++u)
            {
                const int m = m0 + u * T;
                z[u]        = src8 ? reinterpret_cast<const float2 *>(src)[m]
                                   : make_float2(src[2 * m], src[2 * m + 1]);
                w[u]        = need_w ? twg[C::TW_PRE + m] : make_float2(1.0f, 0.0f);     /* w_M^m */
            }
            #pragma unroll
            for (int u = 0; u < LB; ++u)
            {
                const int m = m0 + u * T;
                float2 zb   = cmul(z[u], w[u]);
                if (NH == 2)    { A[m] = z[u]; A[P + m] = zb; }
                else            { A[m] = (pass == 0) ? z[u] : zb; }
            }
        }
        __syncthreads();

        CHAIN_STAMP(4096 + blockIdx.x, 2);
        const float2 *R = fft_smem<RANK, false, PP, TT, WM, true, NHO, TWC>(A, B, tw, tid);
        CHAIN_STAMP(4096 + blockIdx.x, 3);
        if (SMEM_OUT)
        {
            out         = (R == A) ? B : A;
            *smem_out   = out;
        }

        /* split post-pass over pairs (k, M-k), k = 0 .. M/2; thread 0 takes k = 0 and k = M/2.
         * One resident half: only the bins k = 2 i + pass of its parity. */
        constexpr int KSTEP = (NH == 2) ? 1 : 2;
        constexpr int KN    = (M / 2) / KSTEP;                  /* bins visited per pass */
        constexpr int LK    = (KN / T >= 8) ? 8 : ((KN / T >= 1) ? (KN / T) : 1);
        #pragma unroll 1
        for (int i0 = tid; i0 < KN; i0 += LK * T)
        {
            float2 w[LK];
            #pragma unroll
            for (int u = 0; u < LK; ++u)
            {
                const int k = (i0 + u * T) * KSTEP + ((NH == 2) ? 0 : pass);
                w[u]        = (i0 + u * T < KN) ? twx[C::TW_POST + k] : make_float2(0.0f, 0.0f);
            }
            #pragma unroll
            for (int u = 0; u < LK; ++u)
            {
                if (i0 + u * T >= KN)
                    continue;
                const int k = (i0 + u * T) * KSTEP + ((NH == 2) ? 0 : pass);
                if (k == 0)
                {
                    float2 z0   = R[0];                         /* Z[0]: (DC, Nyquist) */
                    out[0]      = make_float2(z0.x + z0.y, z0.x - z0.y);
                    float2 zh   = R[P / 2];                     /* Z[M/2] pairs with itself: X = conj(Z) */
                    out[M / 2]  = make_float2(zh.x, -zh.y);
                    continue;
                }
                const int par = k & 1;
                const float2 *half  = R + ((NH == 2) ? par * P : 0);
                int ik      = k >> 1;
                int im      = par ? (P - 1 - ik) : (P - ik);
                float2 zk   = half[ik], zm = half[im];
                /* e = (zk + conj(zm))/2 ; o = (zk - conj(zm))/2 ; X[k] = e - i w^k o */
                float2 e    = make_float2(0.5f * (zk.x + zm.x), 0.5f * (zk.y - zm.y));
                float2 o    = make_float2(0.5f * (zk.x - zm.x), 0.5f * (zk.y + zm.y));
                float2 wo   = cmul(w[u], o);
                out[k]      = make_float2(e.x + wo.y, e.y - wo.x);
                /* X[M-k] = conj(e) - i conj(w) conj(o) = conj(e) - i conj(wo) */
                out[M - k]  = make_float2(e.x - wo.y, -e.y - wo.x);
            }
        }
        if (NH == 1)
            __syncthreads();
    }
}

/* copies the r = 1 third of every radix-4 pass of the global table into the compact shared-memory one */
template <typename C>
__device__ __forceinline__ void stage_compact_twiddles(float2 *twc, const float2 *twg, int tid)
{
    /* entry e of the compact table is entry pass_base(e) * 3 + (e - pass_base(e)) ... walked flat so
     * that a thread's loads are independent of each other (all in flight at once) */
    constexpr int LT = 4;
    #pragma unroll 1
    for (int e0 = tid; e0 < C::TWC_N; e0 += LT * C::T)
    {
        float2 v[LT];
        int at[LT];
        #pragma unroll
        for (int u = 0; u < LT; ++u)
        {
            const int e = e0 + u * C::T;
            /* pass with Ns entries starts at compact offset (Ns - NS0) / 3: Ns = the largest
             * NS0 * 4^j with (Ns - NS0) / 3 <= e */
            int Ns = C::NS0;
            while ((4 * Ns - C::NS0) / 3 <= e)
                Ns <<= 2;
            at[u]       = e;
            v[u]        = (e < C::TWC_N) ? twg[(Ns - C::NS0) + (e - (Ns - C::NS0) / 3)] : make_float2(0.0f, 0.0f);
        }
        #pragma unroll
        for (int u = 0; u < LT; ++u)
            if (at[u] < C::TWC_N)
                twc[at[u]]  = v[u];
    }
}

template <int RANK>
__global__ void __launch_bounds__(FftCfg<RANK>::T)
k_fwd(const StepArgs a)
{
    using C = FftCfg<RANK>;
    extern __shared__ float2 sm[];
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    float2 *A               = sm;
    float2 *B               = C::PP ? sm + C::WORK : nullptr;
    const float2 *tw        = a.tw;
    if (C::TWS)
    {
        float2 *tws         = sm + C::WORK * (C::PP ? 2 : 1);
        for (int i = threadIdx.x; i < C::TW_TOTAL; i += C::T)
            tws[i]              = a.tw[i];
        tw                  = tws;
        __syncthreads();
    }
    else
    {
        float2 *twc         = sm + C::WORK;
        stage_compact_twiddles<C>(twc, a.tw, threadIdx.x);
        tw                  = twc;
        __syncthreads();
    }
    /* (three-kernel path with programmatic serialisation: the table staging above overlaps the
     * previous launch; everything below reads what earlier launches wrote -- unless the host knows
     * that no launch in flight writes the input block, STEP_EARLY_SRC: then the transform runs under
     * the MAC that was launched ahead, and one CTA waits at the very end for completion order) */
    const bool early_src = (a.flags & STEP_EARLY_SRC) != 0;
    if (!early_src)
        asm volatile("griddepcontrol.wait;" ::: "memory");
    /* grid-stride over the jobs: a launch over many frames (IR ingest, multi-frame calls) keeps
     * one resident set of CTAs and stages the twiddle table once per CTA; these launches are
     * throughput-bound, so every twiddle comes from the shared-memory copy (one load per butterfly) */
    for (uint32_t j = blockIdx.x; j < a.n_jobs; j += gridDim.x)
    {
        const Job job           = fetch_job(a, j);
        fwd_body<RANK, C::PP, 0, false, true, 0, !C::TWS>(A, B, job.src, job.spec, a.tw, tw, threadIdx.x);
        __syncthreads();            /* the work buffers are reused by the next job */
    }
    if (early_src && (blockIdx.x == 0) && (threadIdx.x == 0))
        asm volatile("griddepcontrol.wait;" ::: "memory");
}

/* k_fwd_half : ranks 13..16 with few frames per launch.  One CTA transforms a whole frame in k_fwd,
 * so 64 instances keep 64 of 148 SMs busy (and at rank 16, where only one half fits in shared
 * memory, run the two halves one after the other).  The even and odd bins are independent all the
 * way to the output row, so here work item w = (job w / 2, half w % 2) gets a CTA of its own. */
template <int RANK>
__global__ void __launch_bounds__(FftCfg<RANK, 0, 1>::T)
k_fwd_half(const StepArgs a)
{
    using C = FftCfg<RANK, 0, 1>;
    static_assert(!C::PP && !C::TWS, "k_fwd_half: ranks 13..16");
    extern __shared__ float2 sm[];
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    float2 *twc             = sm + C::WORK;
    stage_compact_twiddles<C>(twc, a.tw, threadIdx.x);
    __syncthreads();
    const bool early_src = (a.flags & STEP_EARLY_SRC) != 0;     /* see k_fwd */
    if (!early_src)
        asm volatile("griddepcontrol.wait;" ::: "memory");
    CHAIN_STAMP(4096 + blockIdx.x, 0);
    for (uint32_t w = blockIdx.x; w < 2 * a.n_jobs; w += gridDim.x)
    {
        const Job job           = fetch_job(a, w >> 1);
        fwd_body<RANK, false, 0, false, true, 1, true>(sm, nullptr, job.src, job.spec, a.tw, twc, threadIdx.x,
                                                       nullptr, int(w & 1u));
        __syncthreads();
    }
    CHAIN_STAMP(4096 + blockIdx.x, 1);
    if (early_src && (blockIdx.x == 0) && (threadIdx.x == 0))
        asm volatile("griddepcontrol.wait;" ::: "memory");
}

/* ------------------------------------------------------------------------------------------- */
/* inv_body : sums the MAC's partial rows, merges the packed spectrum back into the P-point      */
/* even/odd sub-sequences, runs two inverse FFTs and combines only the first F of the 2F output  */
/* samples (the second half is time-aliased garbage in the folded-overlap form).  `full` also    */
/* emits samples [F, 2F) (used by the fastconv primitives).                                      */

/* MODE bit 0 (INV_OLA, needs `full` and an 8-byte aligned dst of 2F floats): overlap-add with a
 * shift, dst[j] = dst[j + F] + y[j], dst[j + F] = y[j + F] (Equalizer.cpp:482-484);
 * MODE bit 1 (INV_PRESUMMED, ping-pong ranks): B already holds the spectrum, yp / splits unused;
 * MODE bit 2 (INV_STAGED, ping-pong ranks): yp is ONE spectrum row in shared memory. */
enum { INV_OLA = 1, INV_PRESUMMED = 2, INV_STAGED = 4 };

template <int RANK, bool PP, int RG = 8, int TT = 0, int MODE = 0, bool WM = (RANK >= 12), int NHO = 0, bool TWC = false>     /* RG: partial rows loaded per round (registers) */
__device__ __forceinline__ void inv_body(float2 *A, float2 *B, const float2 *yp, uint32_t splits,
                                         float *dst, const float2 *twg, const float2 *tw, bool full, int tid,
                                         int only_pass = -1, const float2 *g0 = nullptr, const float2 *x0 = nullptr,
                                         const float2 *yp2 = nullptr, uint32_t splits2 = 0)
{
    /* yp2, splits2: more rows to add after the `splits` rows of yp (k_frame lookahead: the block's T rows) */
    /* g0, x0 (rows summed from global memory only, !PP): one more term, g0[k] * x0[k] -- partition 0
     * against the block's own spectrum (STEP_Q0_IN_INV); bin 0 packs two real values (DC, Nyquist) */
    const float2 *twx       = TWC ? twg : tw;      /* TWC: `tw` is the compact pass table (fft_smem) */
    /* only_pass (one resident half, NH == 1; k_inv_half): 0 = the odd bins' half, 1 = the even
     * bins' half; either way dst receives that half's F scaled samples and nothing is combined */
    static_assert((!(MODE & INV_PRESUMMED)) || PP, "inv_body: INV_PRESUMMED needs the second work buffer");
    using C = FftCfg<RANK, TT, NHO>;
    constexpr int P = C::P, M = C::M, T = C::T, NH = C::NH, N = C::N;
    constexpr int ITER = (M / 2) / T;           /* bins k = tid + it*T handled by this thread; even */
    static_assert((ITER >= 2) && ((ITER & 1) == 0), "inv_body: two bins per round");
    const float scale       = 1.0f / float(N);

    #pragma unroll 1
    for (int pass = 0; pass < 2 / NH; ++pass)
    {
        if ((only_pass >= 0) && (pass != only_pass))
            continue;
        /* with one resident half the odd half goes first and is parked in dst */
        const int want = (NH == 1) ? (1 - pass) : 0;

        if (PP && !(MODE & (INV_PRESUMMED | INV_STAGED)))
        {
            /* Reduce the partial rows first, as coalesced float4 columns, into the second work
             * buffer.  The loads are volatile asm so that a whole group is in flight before the
             * first add: this is the exposed tail of the launch. */
            float4 *ysum = reinterpret_cast<float4 *>(B);
            #pragma unroll 1
            for (int c0 = 0; c0 < M / 2; c0 += 2 * T)
            {
                const int ca = c0 + tid, cb = c0 + T + tid;
                float4 sa = make_float4(0.0f, 0.0f, 0.0f, 0.0f), sb = sa;
                #pragma unroll 1
                for (int set = 0; set < 2; ++set)
                {
                const float2 *yr    = set ? yp2 : yp;
                const uint32_t nr   = set ? splits2 : splits;
                for (uint32_t s0 = 0; s0 < nr; s0 += RG)
                {
                    float4 va[RG], vb[RG];
                    #pragma unroll
                    for (int r = 0; r < RG; ++r)
                    {
                        uint32_t row = min(s0 + r, nr - 1);         /* clamp: the extra loads are dropped below */
                        const float4 *rp = reinterpret_cast<const float4 *>(yr + uint64_t(row) * M);
                        va[r]       = ld_cg_f4(rp + ca);
                        vb[r]       = ld_cg_f4(rp + cb);
                    }
                    #pragma unroll
                    for (int r = 0; r < RG; ++r)
                    {
                        if (s0 + r < nr)
                        {
                            sa.x += va[r].x; sa.y += va[r].y; sa.z += va[r].z; sa.w += va[r].w;
                            sb.x += vb[r].x; sb.y += vb[r].y; sb.z += vb[r].z; sb.w += vb[r].w;
                        }
                    }
                }
                }
                ysum[ca]    = sa;
                ysum[cb]    = sb;
            }
            __syncthreads();
        }

        /* UB bins per round, each with its mirror (k = 0 pairs with M/2: both self-paired specials
         * ride in thread 0's first slot).  One resident half visits only the bins k = 2 i + want of
         * its parity.  Without a second work buffer (ranks >= 13, one CTA per SM) the partial rows and
         * the twiddles come straight from global memory / L2: eight bins per round keep enough loads
         * in flight to cover that latency. */
        constexpr int KSTEP     = (NH == 2) ? 1 : 2;
        constexpr int ROUNDS    = ITER / KSTEP;
        constexpr int UB        = PP ? 2 : ((ROUNDS >= 8) ? 8 : ROUNDS);
        static_assert((ROUNDS >= 1) && (ROUNDS % UB == 0), "inv_body: whole rounds");
        #pragma unroll 1
        for (int it0 = 0; it0 < ROUNDS; it0 += UB)
        {
            int k[UB], km[UB];
            float2 wk[UB];
            #pragma unroll
            for (int u = 0; u < UB; ++u)
            {
                k[u]        = (tid + (it0 + u) * T) * KSTEP + ((NH == 2) ? 0 : want);
                km[u]       = (k[u] == 0) ? (M / 2) : (M - k[u]);
                wk[u]       = twg[C::TW_POST + k[u]];
            }
            float2 yk[UB], ym[UB];
            if (PP)
            {
                const float2 *Y = (MODE & INV_STAGED) ? yp : B;
                #pragma unroll
                for (int u = 0; u < UB; ++u)
                {
                    yk[u]       = Y[k[u]];
                    ym[u]       = Y[km[u]];
                }
            }
            else
            {
                #pragma unroll
                for (int u = 0; u < UB; ++u)
                    yk[u] = ym[u] = make_float2(0.0f, 0.0f);
                for (uint32_t s = 0; s < splits + splits2; ++s)
                {
                    const float2 *row = (s < splits) ? yp + uint64_t(s) * M : yp2 + uint64_t(s - splits) * M;
                    #pragma unroll
                    for (int u = 0; u < UB; ++u)
                    {
                        yk[u]       = cadd(yk[u], __ldcg(row + k[u]));
                        ym[u]       = cadd(ym[u], __ldcg(row + km[u]));
                    }
                }
                if (g0 != nullptr)
                {
                    float2 gk[UB], xk[UB], gm[UB], xm[UB];
                    #pragma unroll
                    for (int u = 0; u < UB; ++u)
                    {
                        gk[u]       = __ldcg(g0 + k[u]);
                        xk[u]       = __ldcg(x0 + k[u]);
                        gm[u]       = __ldcg(g0 + km[u]);
                        xm[u]       = __ldcg(x0 + km[u]);
                    }
                    #pragma unroll
                    for (int u = 0; u < UB; ++u)
                    {
                        yk[u]       = cadd(yk[u], (k[u] == 0) ? make_float2(gk[u].x * xk[u].x, gk[u].y * xk[u].y) : cmul(gk[u], xk[u]));
                        ym[u]       = cadd(ym[u], cmul(gm[u], xm[u]));
                    }
                }
            }

            #pragma unroll
            for (int u = 0; u < UB; ++u)
            {
                int par     = k[u] & 1;
                float2 *half = A + ((NH == 2) ? par * P : 0);
                if (k[u] == 0)
                {
                    /* (DC, Nyquist) -> Z[0] = (DC + Ny) + i (DC - Ny);  Z[M/2] = 2 conj(Y[M/2]) */
                    half[0]     = make_float2(yk[u].x + yk[u].y, yk[u].x - yk[u].y);
                    half[P / 2] = make_float2(2.0f * ym[u].x, -2.0f * ym[u].y);
                    continue;
                }
                /* e = yk + conj(ym) ; o = conj(w^k) (yk - conj(ym)) ; Z[k] = e + i o ; Z[M-k] = conj(e) + i conj(o) */
                float2 e    = make_float2(yk[u].x + ym[u].x, yk[u].y - ym[u].y);
                float2 df   = make_float2(yk[u].x - ym[u].x, yk[u].y + ym[u].y);
                float2 o    = cmulc(df, wk[u]);
                int ik      = k[u] >> 1;
                int im      = par ? (P - 1 - ik) : (P - ik);
                half[ik]    = make_float2(e.x - o.y, e.y + o.x);
                half[im]    = make_float2(e.x + o.y, o.x - e.y);
            }
        }
        __syncthreads();

        CHAIN_STAMP(4096 + 512 + blockIdx.x, 2);
        const float2 *R = fft_smem<RANK, true, PP, TT, WM, true, NHO, TWC>(A, B, tw, tid);
        CHAIN_STAMP(4096 + 512 + blockIdx.x, 3);

        /* z[m] = (A[m] + conj(w_M^m) B[m]) / N ; z[m + P] = (A[m] - conj(w_M^m) B[m]) / N
         * (global loads -- the twiddle, the parked half -- LBO at a time before the first use) */
        constexpr int LBO = (P / T >= 8) ? 8 : (P / T);
        const bool need_w   = (NH == 2) || (pass == 0);
        const bool need_pk  = (NH == 1) && (pass != 0) && (only_pass != 1);
        #pragma unroll 1
        for (int m0 = tid; m0 < P; m0 += LBO * T)
        {
        float2 wv[LBO], pkv[LBO];
        #pragma unroll
        for (int u = 0; u < LBO; ++u)
        {
            const int m = m0 + u * T;
            wv[u]       = need_w ? twx[C::TW_PRE + m] : make_float2(1.0f, 0.0f);
            pkv[u]      = need_pk ? make_float2(dst[2 * m], dst[2 * m + 1]) : make_float2(0.0f, 0.0f);
        }
        #pragma unroll
        for (int u = 0; u < LBO; ++u)
        {
            const int m = m0 + u * T;
            float2 lo, hi;
            if (NH == 2)
            {
                float2 av   = R[m];
                float2 bv   = cmulc(R[P + m], wv[u]);
                lo          = make_float2((av.x + bv.x) * scale, (av.y + bv.y) * scale);
                hi          = make_float2((av.x - bv.x) * scale, (av.y - bv.y) * scale);
            }
            else if (pass == 0)
            {
                /* park conj(w) B / N where the result will go; the same thread reads it back */
                float2 bv   = cmulc(R[m], wv[u]);
                dst[2 * m]      = bv.x * scale;
                dst[2 * m + 1]  = bv.y * scale;
                continue;
            }
            else if (only_pass == 1)
            {
                dst[2 * m]      = R[m].x * scale;
                dst[2 * m + 1]  = R[m].y * scale;
                continue;
            }
            else
            {
                float2 av   = R[m];
                float2 pk   = pkv[u];
                lo          = make_float2(av.x * scale + pk.x, av.y * scale + pk.y);
                hi          = make_float2(av.x * scale - pk.x, av.y * scale - pk.y);
            }

            if (MODE & INV_OLA)
            {
                float2 tail = reinterpret_cast<const float2 *>(dst)[m + P];
                reinterpret_cast<float2 *>(dst)[m]      = make_float2(tail.x + lo.x, tail.y + lo.y);
                reinterpret_cast<float2 *>(dst)[m + P]  = hi;
            }
            else if ((reinterpret_cast<uintptr_t>(dst) & 7) == 0)
            {
                reinterpret_cast<float2 *>(dst)[m]  = lo;
                if (full)
                    reinterpret_cast<float2 *>(dst)[m + P]  = hi;
            }
            else
            {
                dst[2 * m]      = lo.x;
                dst[2 * m + 1]  = lo.y;
                if (full)
                {
                    dst[2 * (m + P)]        = hi.x;
                    dst[2 * (m + P) + 1]    = hi.y;
                }
            }
        }
        }
        if (NH == 1)
            __syncthreads();
    }
}

/* RG = 2 serves launches with one or two partial rows per job (multi-frame calls, the fastconv
 * primitives): few registers, so that as many CTAs as shared memory allows are resident. */
template <int RANK, int RG>
struct InvCfg
{
    static constexpr int MINB = (RG > 2) ? 0 : (RANK == 11) ? 5 : (RANK == 12) ? 2 : 0;     /* 0: left to the compiler */
};

template <int RANK, int RG = 8>
__global__ void __launch_bounds__(FftCfg<RANK>::T, InvCfg<RANK, RG>::MINB)
k_inv(const StepArgs a)
{
    using C = FftCfg<RANK>;
    extern __shared__ float2 sm[];
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    float2 *A               = sm;
    float2 *B               = C::PP ? sm + C::WORK : nullptr;
    const float2 *tw        = a.tw;
    if (C::TWS)
    {
        float2 *tws         = sm + C::WORK * (C::PP ? 2 : 1);
        for (int i = threadIdx.x; i < C::TW_TOTAL; i += C::T)
            tws[i]              = a.tw[i];
        tw                  = tws;
        __syncthreads();
    }
    else
    {
        float2 *twc         = sm + C::WORK;
        stage_compact_twiddles<C>(twc, a.tw, threadIdx.x);
        tw                  = twc;
        __syncthreads();
    }
    asm volatile("griddepcontrol.wait;" ::: "memory");     /* the partial rows of the launch before */
    if ((a.flags & STEP_Q0_IN_INV) && (a.chain_head != nullptr) && (blockIdx.x == 0) && (threadIdx.x == 0))
        asm volatile("st.release.gpu.global.u32 [%0], %1;" :: "l"(a.chain_head), "r"(uint32_t(a.t_base + a.frame0) + 1u) : "memory");
    for (uint32_t j = blockIdx.x; j < a.n_jobs; j += gridDim.x)
    {
        const Job job           = fetch_job(a, j);
        const float2 *g0        = nullptr;
        if ((!C::PP) && (a.flags & STEP_Q0_IN_INV))
        {
            const InstDesc &d       = a.inst[job.inst];
            if ((d.q_lo == 0) && (d.nq > 0))
                g0                      = d.G;          /* row 0 = partition 0 */
        }
        inv_body<RANK, C::PP, RG, 0, 0, true, 0, !C::TWS>(A, B, a.ypart + uint64_t(j) * rows_per_job(a) * C::M, rows_per_job(a),
                                                          job.dst, a.tw, tw, (a.flags & INV_FULL) != 0, threadIdx.x, -1, g0, job.spec);
        __syncthreads();
    }
}

/* k_inv_half + k_inv_combine : the inverse transform of ranks 13..16 with few frames per launch,
 * one CTA per HALF frame (see k_fwd_half).  The halves meet only in the last pass,
 * y[j] = e[j] + o[j], y[j + F] = e[j] - o[j], so each CTA leaves its F scaled samples in
 * park[job][half] and an element-wise launch combines them. */
template <int RANK>
__global__ void __launch_bounds__(FftCfg<RANK, 0, 1>::T)
k_inv_half(const StepArgs a, uint32_t *tickets)
{
    __shared__ uint32_t last;
    using C = FftCfg<RANK, 0, 1>;
    static_assert(!C::PP && !C::TWS, "k_inv_half: ranks 13..16");
    extern __shared__ float2 sm[];
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    float2 *twc             = sm + C::WORK;
    stage_compact_twiddles<C>(twc, a.tw, threadIdx.x);
    __syncthreads();
    CHAIN_STAMP(4096 + 512 + blockIdx.x, 0);
    asm volatile("griddepcontrol.wait;" ::: "memory");
    CHAIN_STAMP(4096 + 512 + blockIdx.x, 1);
    if ((a.flags & STEP_Q0_IN_INV) && (a.chain_head != nullptr) && (blockIdx.x == 0) && (threadIdx.x == 0))
        asm volatile("st.release.gpu.global.u32 [%0], %1;" :: "l"(a.chain_head), "r"(uint32_t(a.t_base + a.frame0) + 1u) : "memory");
    const uint32_t rows = rows_per_job(a);
    for (uint32_t w = blockIdx.x; w < 2 * a.n_jobs; w += gridDim.x)
    {
        const uint32_t j = w >> 1, half = w & 1u;       /* half 0: odd bins, half 1: even bins */
        const float2 *g0 = nullptr, *x0 = nullptr;
        if (a.flags & STEP_Q0_IN_INV)
        {
            const Job jq            = fetch_job(a, j);
            const InstDesc &d       = a.inst[jq.inst];
            if ((d.q_lo == 0) && (d.nq > 0))
                g0                      = d.G;          /* row 0 = partition 0 */
            x0                      = jq.spec;
        }
        inv_body<RANK, false, 8, 0, 0, true, 1, true>(sm, nullptr, a.ypart + uint64_t(j) * rows * C::M, rows,
                                                      a.park + (uint64_t(j) * 2 + half) * C::M, a.tw, twc, false,
                                                      threadIdx.x, int(half), g0, x0);
        if (tickets != nullptr)
        {
            /* the second half of a frame to finish combines: y[i] = e[i] + o[i] (and e[i] - o[i] for
             * the upper half of a full inverse) -- no separate element-wise launch */
            __threadfence();
            __syncthreads();
            if (threadIdx.x == 0)
            {
                const uint32_t old  = atomicAdd(&tickets[j], 1u);
                last                = (old == 1u) ? 1u : 0u;
                if (last)
                    tickets[j]          = 0;
            }
            __syncthreads();
            if (last)
            {
                __threadfence();
                const Job job       = fetch_job(a, j);
                const bool full     = (a.flags & INV_FULL) != 0;
                const float4 *o4    = reinterpret_cast<const float4 *>(a.park + uint64_t(j) * 2 * C::M);
                const float4 *e4    = o4 + C::M / 4;
                const bool al       = (reinterpret_cast<uintptr_t>(job.dst) & 15) == 0;
                /* CB columns per round, all loads in flight before the first store (one round trip to
                 * L2 per round instead of one per column: this loop is the exposed end of the block) */
                constexpr uint32_t COLS = uint32_t(C::M) / 4 / C::T;
                constexpr uint32_t CB   = (COLS % 4 == 0) ? 4 : ((COLS % 2 == 0) ? 2 : 1);
                static_assert(COLS * C::T * 4 == uint32_t(C::M), "k_inv_half: whole columns per thread");
                #pragma unroll 1
                for (uint32_t c0 = 0; c0 < COLS; c0 += CB)
                {
                    float4 ev[CB], ov[CB];
                    #pragma unroll
                    for (uint32_t u = 0; u < CB; ++u)
                    {
                        const uint32_t i    = threadIdx.x + (c0 + u) * C::T;
                        ev[u]               = ld_cg_f4(e4 + i);
                        ov[u]               = ld_cg_f4(o4 + i);
                    }
                    #pragma unroll
                    for (uint32_t u = 0; u < CB; ++u)
                    {
                        const uint32_t i    = threadIdx.x + (c0 + u) * C::T;
                        const float4 lo = make_float4(ev[u].x + ov[u].x, ev[u].y + ov[u].y, ev[u].z + ov[u].z, ev[u].w + ov[u].w);
                        const float4 hi = make_float4(ev[u].x - ov[u].x, ev[u].y - ov[u].y, ev[u].z - ov[u].z, ev[u].w - ov[u].w);
                        if (al)
                        {
                            reinterpret_cast<float4 *>(job.dst)[i]  = lo;
                            if (full)
                                reinterpret_cast<float4 *>(job.dst)[C::M / 4 + i] = hi;
                        }
                        else
                        {
                            job.dst[4 * i] = lo.x; job.dst[4 * i + 1] = lo.y; job.dst[4 * i + 2] = lo.z; job.dst[4 * i + 3] = lo.w;
                            if (full)
                            {
                                float *d2 = job.dst + C::M;
                                d2[4 * i] = hi.x; d2[4 * i + 1] = hi.y; d2[4 * i + 2] = hi.z; d2[4 * i + 3] = hi.w;
                            }
                        }
                    }
                }
            }
        }
        __syncthreads();
    }
    CHAIN_STAMP(4096 + 512 + blockIdx.x, 4);
}

__global__ void k_inv_combine(const StepArgs a)
{
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");
    const uint32_t F    = 1u << (a.rank - 1);
    const bool full     = (a.flags & INV_FULL) != 0;
    for (uint32_t j = blockIdx.y; j < a.n_jobs; j += gridDim.y)
    {
        const Job job       = fetch_job(a, j);
        const float *o      = a.park + uint64_t(j) * 2 * F;
        const float *e      = o + F;
        for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < F; i += gridDim.x * blockDim.x)
        {
            float ev = e[i], ov = o[i];
            job.dst[i]          = ev + ov;
            if (full)
                job.dst[F + i]      = ev - ov;
        }
    }
}

/* ------------------------------------------------------------------------------------------- */
/* k_mac : the roofline kernel.  Y[job][split][k] = sum_{q in chunk} G_q[k] * X_{t-q}[k].        */
/*                                                                                             */
/* Pure fp32 stream: 16 bytes in per complex MAC, no reuse (one frame per call), so the only job */
/* is to keep enough bytes in flight.  One elected thread feeds an NS-deep shared-memory ring     */
/* with 1-D TMA bulk copies (cp.async.bulk + mbarrier complete_tx); all threads drain it with     */
/* conflict-free LDS.128 and FFMA.  No tensor cores: 0.5 flop/byte is far below any MMA ridge.    */
/*                                                                                             */
/* grid = (jobs * splits, M / TB).  Stage = QB consecutive partitions x TB bins of G and of the   */
/* ring (QB > 1 only when TB == M, where consecutive rows are contiguous in memory).             */

__device__ __forceinline__ uint32_t smem_u32(const void *p)
{
    return uint32_t(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count) : "memory");
}

__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;"
                 :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}

__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
    uint32_t done;
    do
    {
        asm volatile(
            "{\n\t"
            ".reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t"
            "}"
            : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    } while (!done);
}

/* global -> shared bulk copy (TMA, 1-D); bytes % 16 == 0, both addresses 16-byte aligned */
/* IR spectra and ring rows are read once per block and the working set is several times the L2:
 * they are fetched with an evict-first L2 policy so that they do not push out what IS reused
 * (partial rows, the freshly written spectrum, the tables).  Measured on config 3: 67.2 us per
 * block with the hint, 70.0 us without (profiles/README.md). */
__device__ __forceinline__ uint64_t stream_policy()
{
    uint64_t policy;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(policy));
    return policy;
}

/* rows that later launches read again (k_frame lookahead: the head rows q < 2K) */
__device__ __forceinline__ uint64_t keep_policy()
{
    uint64_t policy;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(policy));
    return policy;
}

__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar,
                                         uint64_t policy)
{
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
        :: "r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)), "l"(policy) : "memory");
}

__device__ __forceinline__ void bulk_g2s_plain(void *dst, const void *src, uint32_t bytes, uint64_t *bar)
{
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
        :: "r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

/* ------------------------------------------------------------------------------------------- */
/* k_fwd_staged / k_inv_staged : the transforms of launches that loop over MANY jobs per CTA     */
/* (multi-frame calls, IR ingest, the fastconv primitives) on the ping-pong ranks.  A CTA's      */
/* phases are separated by barriers, so a plain global load at the start of a job is fully       */
/* exposed; here one elected thread fetches the NEXT job's input -- F samples, or one spectrum   */
/* row -- with a TMA bulk copy into a two-slot shared-memory ring while the current job is       */
/* transformed.  Inputs that are not 16-byte aligned are read directly, as in k_fwd / k_inv.     */

template <int RANK>
struct StageCfg
{
    using C = FftCfg<RANK>;
    static constexpr size_t OFF         = (C::SMEM + 127) & ~size_t(127);
    static constexpr size_t FWD_SLOT    = C::M * sizeof(float);
    static constexpr size_t INV_SLOT    = C::M * sizeof(float2);
    static constexpr size_t FWD_SMEM    = OFF + 2 * FWD_SLOT + 2 * sizeof(uint64_t);
    static constexpr size_t INV_SMEM    = OFF + 2 * INV_SLOT + 2 * sizeof(uint64_t);
    static constexpr int    INV_MINB    = (RANK == 11) ? 5 : (RANK == 12) ? 2 : 0;
};

__device__ __forceinline__ bool tma_aligned(const void *p)
{
    return (reinterpret_cast<uintptr_t>(p) & 15) == 0;
}

template <int RANK>
__global__ void __launch_bounds__(FftCfg<RANK>::T)
k_fwd_staged(const StepArgs a)
{
    using C = FftCfg<RANK>;
    using S = StageCfg<RANK>;
    static_assert(C::PP && C::TWS, "k_fwd_staged: ping-pong ranks only");
    extern __shared__ __align__(128) unsigned char st_sm[];
    float2 *A               = reinterpret_cast<float2 *>(st_sm);
    float2 *B               = A + C::WORK;
    float2 *tws             = A + 2 * C::WORK;
    float *slots            = reinterpret_cast<float *>(st_sm + S::OFF);
    uint64_t *bars          = reinterpret_cast<uint64_t *>(st_sm + S::OFF + 2 * S::FWD_SLOT);
    const int tid           = threadIdx.x;

    for (int i = tid; i < C::TW_TOTAL; i += C::T)
        tws[i]                  = a.tw[i];
    uint32_t j              = blockIdx.x;
    Job job;
    memset(&job, 0, sizeof(job));
    if (j < a.n_jobs)
        job                     = fetch_job(a, j);
    if (tid == 0)
    {
        mbar_init(&bars[0], 1);
        mbar_init(&bars[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        if ((j < a.n_jobs) && tma_aligned(job.src))
        {
            mbar_expect_tx(&bars[0], uint32_t(S::FWD_SLOT));
            bulk_g2s_plain(slots, job.src, uint32_t(S::FWD_SLOT), &bars[0]);
        }
    }
    __syncthreads();

    uint32_t ph0 = 0, ph1 = 0;
    for (uint32_t it = 0; j < a.n_jobs; ++it, j += gridDim.x)
    {
        const uint32_t s        = it & 1u;
        Job next                = job;
        const bool more         = (j + gridDim.x < a.n_jobs);
        if (more)
            next                    = fetch_job(a, j + gridDim.x);
        if ((tid == 0) && more && tma_aligned(next.src))
        {
            /* slot s ^ 1 was last read by the job before this one; a barrier lies in between */
            mbar_expect_tx(&bars[s ^ 1u], uint32_t(S::FWD_SLOT));
            bulk_g2s_plain(slots + (s ^ 1u) * C::M, next.src, uint32_t(S::FWD_SLOT), &bars[s ^ 1u]);
        }
        const float *src        = job.src;
        if (tma_aligned(job.src))
        {
            if (s)  { mbar_wait(&bars[1], ph1); ph1 ^= 1u; }
            else    { mbar_wait(&bars[0], ph0); ph0 ^= 1u; }
            src                     = slots + s * C::M;
        }
        fwd_body<RANK, true, 0, false, true>(A, B, src, job.spec, tws, tws, tid);
        __syncthreads();            /* work buffers and the slot are reused */
        job                     = next;
    }
}

template <int RANK>
__global__ void __launch_bounds__(FftCfg<RANK>::T, StageCfg<RANK>::INV_MINB)
k_inv_staged(const StepArgs a)     /* one partial row per job */
{
    using C = FftCfg<RANK>;
    using S = StageCfg<RANK>;
    static_assert(C::PP && C::TWS, "k_inv_staged: ping-pong ranks only");
    extern __shared__ __align__(128) unsigned char st_sm[];
    float2 *A               = reinterpret_cast<float2 *>(st_sm);
    float2 *B               = A + C::WORK;
    float2 *tws             = A + 2 * C::WORK;
    float2 *slots           = reinterpret_cast<float2 *>(st_sm + S::OFF);
    uint64_t *bars          = reinterpret_cast<uint64_t *>(st_sm + S::OFF + 2 * S::INV_SLOT);
    const int tid           = threadIdx.x;
    const bool full         = (a.flags & INV_FULL) != 0;

    for (int i = tid; i < C::TW_TOTAL; i += C::T)
        tws[i]                  = a.tw[i];
    uint32_t j              = blockIdx.x;
    if (tid == 0)
    {
        mbar_init(&bars[0], 1);
        mbar_init(&bars[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        if (j < a.n_jobs)
        {
            mbar_expect_tx(&bars[0], uint32_t(S::INV_SLOT));
            bulk_g2s_plain(slots, a.ypart + uint64_t(j) * C::M, uint32_t(S::INV_SLOT), &bars[0]);
        }
    }
    __syncthreads();

    uint32_t ph0 = 0, ph1 = 0;
    for (uint32_t it = 0; j < a.n_jobs; ++it, j += gridDim.x)
    {
        const uint32_t s        = it & 1u;
        const Job job           = fetch_job(a, j);
        if ((tid == 0) && (j + gridDim.x < a.n_jobs))
        {
            mbar_expect_tx(&bars[s ^ 1u], uint32_t(S::INV_SLOT));
            bulk_g2s_plain(slots + (s ^ 1u) * C::M, a.ypart + uint64_t(j + gridDim.x) * C::M, uint32_t(S::INV_SLOT),
                           &bars[s ^ 1u]);
        }
        if (s)  { mbar_wait(&bars[1], ph1); ph1 ^= 1u; }
        else    { mbar_wait(&bars[0], ph0); ph0 ^= 1u; }
        inv_body<RANK, true, 2, 0, INV_STAGED, true>(A, B, slots + s * C::M, 1, job.dst, tws, tws, full, tid);
        __syncthreads();
    }
}

struct MacShape
{
    uint32_t TB;        /* bins per CTA tile                 */
    uint32_t QB;        /* partitions per stage              */
    uint32_t NS;        /* stages                            */
    uint32_t bias;      /* k_frame: partitions taken off split 0, which also transforms the input */
};

/* Partition chunk [c0, c1) (relative to the job's first partition) of split `split`. */
__host__ __device__ __forceinline__ void chunk_range(uint32_t nq, uint32_t split, uint32_t splits, uint32_t bias,
                                            uint32_t &c0, uint32_t &c1)
{
    uint32_t even   = nq / splits;
    if (nq < splits)
    {
        /* one partition each for the first nq splits: split 0 always owns partition 0 */
        c0          = min(split, nq);
        c1          = min(split + 1, nq);
        return;
    }
    if ((splits <= 1) || (bias == 0) || (even <= bias + 1))
    {
        c0          = uint32_t((uint64_t(nq) * split) / splits);
        c1          = uint32_t((uint64_t(nq) * (split + 1)) / splits);
        return;
    }
    uint32_t len0   = even - bias;
    uint32_t rest   = nq - len0;
    if (split == 0)
    {
        c0          = 0;
        c1          = len0;
        return;
    }
    c0              = len0 + uint32_t((uint64_t(rest) * (split - 1)) / (splits - 1));
    c1              = len0 + uint32_t((uint64_t(rest) * split) / (splits - 1));
}

/* The eager pending MAC (synchronous host callers) has time that the launch which delivers the
 * block has not: the last CTA of a job folds the job's rows into one, in the order the inverse
 * transform would have added them, so that launch sums two rows instead of splits + 1.  Kept out
 * of line: k_mac's register budget (4 CTAs per SM) belongs to the partition stream. */
__device__ __noinline__ void fold_rows(uint32_t *ticket, float2 *job_rows, uint32_t splits, uint32_t n_cta, uint32_t M,
                                       uint32_t tid, uint32_t T)
{
    __shared__ uint32_t fold_last;
    __threadfence();
    __syncthreads();
    if (tid == 0)
    {
        uint32_t old    = atomicAdd(ticket, 1u);
        uint32_t last   = (old == n_cta - 1) ? 1u : 0u;
        if (last)
            *ticket         = 0;
        fold_last       = last;
    }
    __syncthreads();
    if (fold_last == 0)
        return;
    __threadfence();
    float4 *rows    = reinterpret_cast<float4 *>(job_rows);
    const uint32_t C4 = M / 2;                                      /* float4 columns per row */
    for (uint32_t c = tid; c < C4; c += T)
    {
        float4 sum      = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        for (uint32_t s0 = 0; s0 < splits; s0 += 8)
        {
            float4 v[8];
            #pragma unroll
            for (int r = 0; r < 8; ++r)
                v[r]            = ld_cg_f4(rows + uint64_t(min(s0 + r, splits - 1)) * C4 + c);
            #pragma unroll
            for (int r = 0; r < 8; ++r)
                if (s0 + r < splits)
                {
                    sum.x += v[r].x; sum.y += v[r].y; sum.z += v[r].z; sum.w += v[r].w;
                }
        }
        rows[uint64_t(splits - 1) * C4 + c] = sum;
    }
}

constexpr int MAC_VPT = 2;      /* float4 columns per thread; blockDim.x = TB / (2 * MAC_VPT) */

__global__ void __launch_bounds__(256, 4)
k_mac(const StepArgs a, const MacShape sh)
{
    extern __shared__ __align__(128) unsigned char smraw[];

    /* A k_frame launch that follows with the programmatic-serialization attribute (the head-only
     * launch of a synchronous host call after the eager pending MAC) may become resident now: it
     * fetches and transforms its input block, which this launch never touches, and reads these
     * partial rows only after its griddepcontrol.wait.  A no-op for any other successor. */
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

    const uint32_t M        = 1u << (a.rank - 1);
    const uint32_t TB       = sh.TB, QB = sh.QB, NS = sh.NS;
    const uint32_t T        = blockDim.x;
    const uint32_t tid      = threadIdx.x;
    CHAIN_STAMP(blockIdx.x + gridDim.x * blockIdx.y, 0);
    const uint32_t jobi     = blockIdx.x / a.splits;
    const uint32_t split    = blockIdx.x % a.splits;
    const uint32_t tile     = blockIdx.y;

    const uint32_t stage_elems = QB * TB;                           /* float2 per operand per stage */
    float2 *sG              = reinterpret_cast<float2 *>(smraw);
    float2 *sX              = sG + size_t(NS) * stage_elems;
    uint64_t *full          = reinterpret_cast<uint64_t *>(sX + size_t(NS) * stage_elems);

    const Job job           = fetch_job(a, jobi);
    const InstDesc d        = a.inst[job.inst];

    /* this CTA's partition chunk [q0, q1) in global partition indices */
    uint32_t qa             = max(job.qa, d.q_lo);
    uint32_t qb             = min(job.qb, d.q_lo + d.nq);
    uint32_t nq             = (qb > qa) ? (qb - qa) : 0;
    uint32_t c0, c1;
    chunk_range(nq, split, a.splits, 0, c0, c1);
    const uint32_t q0       = qa + c0, q1 = qa + c1;
    const uint32_t n_iter   = (q1 - q0 + QB - 1) / QB;

    const float2 *Gt        = d.G + uint64_t(tile) * TB;            /* row r at Gt + r * M */
    const float2 *Xt        = d.ring + uint64_t(tile) * TB;
    const uint32_t row_bytes = TB * uint32_t(sizeof(float2));
    const uint64_t l2_stream = stream_policy();

    if (tid == 0)
    {
        for (uint32_t s = 0; s < NS; ++s)
            mbar_init(&full[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    __syncthreads();

    /* Stage-ring bookkeeping is incremental (next stage buffer, next partition, next ring slot):
     * no integer division inside the streaming loop.  STEP_AFTER_FWD: the CTAs of split 0 visit
     * their stages in the order 1, 2, ..., n_iter - 1, 0 -- stage 0 holds partition q = 0, whose
     * ring row the k_fwd launch right before this one is still writing. */
    const uint32_t late     = ((a.flags & STEP_AFTER_FWD) && (split == 0) && (n_iter > 0)) ? 1u : 0u;
    const uint32_t slot_q0  = uint32_t((uint64_t(job.slot0) + q0) % d.S);
    uint32_t f_it = 0, f_s = 0, f_q = q0 + late * QB;
    uint32_t f_slot         = slot_q0 + late * QB;
    if (f_slot >= d.S)      f_slot -= d.S;
    auto issue_next = [&]()
    {
        if (late && (f_it == n_iter - 1))
        {
            /* the rotated first stage: every earlier launch (the transform of this block) is complete */
            asm volatile("griddepcontrol.wait;" ::: "memory");
            asm volatile("fence.proxy.async;" ::: "memory");
            f_q             = q0;
            f_slot          = slot_q0;
        }
        uint32_t rows   = min(QB, q1 - f_q);
        float2 *g       = sG + size_t(f_s) * stage_elems;
        float2 *x       = sX + size_t(f_s) * stage_elems;
        mbar_expect_tx(&full[f_s], 2u * rows * row_bytes);
        if (TB == M)
        {
            /* IR rows q .. q+rows-1 are contiguous */
            bulk_g2s(g, Gt + uint64_t(f_q - d.q_lo) * M, rows * row_bytes, &full[f_s], l2_stream);
            /* ring slots (slot0 + q) mod S ascend with q: one copy, or two around the wrap */
            uint32_t n1     = min(rows, d.S - f_slot);
            bulk_g2s(x, Xt + uint64_t(f_slot) * M, n1 * row_bytes, &full[f_s], l2_stream);
            if (n1 < rows)
                bulk_g2s(x + size_t(n1) * TB, Xt, (rows - n1) * row_bytes, &full[f_s], l2_stream);
        }
        else
        {
            /* a bin tile of several partitions per stage (QB > 1 with TB < M): one copy per row */
            for (uint32_t r = 0; r < rows; ++r)
            {
                uint32_t sl     = f_slot + r;
                if (sl >= d.S)  sl -= d.S;
                bulk_g2s(g + size_t(r) * TB, Gt + uint64_t(f_q + r - d.q_lo) * M, row_bytes, &full[f_s], l2_stream);
                bulk_g2s(x + size_t(r) * TB, Xt + uint64_t(sl) * M, row_bytes, &full[f_s], l2_stream);
            }
        }
        ++f_it;
        f_q            += QB;
        f_slot         += QB;
        if (f_slot >= d.S)  f_slot -= d.S;
        if (++f_s == NS)    f_s = 0;
    };

    if (tid == 0)
    {
        if ((a.chain_head != nullptr) && (n_iter > 0))
        {
            wait_ge<false>(a.chain_head, uint32_t(a.t_base + a.frame0), a.error, SPIN_ERR_RING);
            asm volatile("fence.proxy.async;" ::: "memory");
        }
        if ((a.flags & STEP_WAIT_HEAD) && (n_iter > 0))
        {
            /* The eager pending MAC of a synchronous caller starts while the k_frame launch that
             * delivers the previous block is still running: partitions q >= q0 >= 1 of block t need
             * the spectra of frames <= t - q0, the newest of which that launch is publishing. */
            wait_ge<false>(a.ring_head + job.inst, job.tlo - q0 + 1u, a.error, SPIN_ERR_RING);
            asm volatile("fence.proxy.async;" ::: "memory");
        }
        while ((f_it < NS) && (f_it < n_iter))
            issue_next();
    }

    float4 acc[MAC_VPT];
    #pragma unroll
    for (int v = 0; v < MAC_VPT; ++v)
        acc[v]      = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    float dny       = 0.0f;         /* sum of Im*Im of the thread's first bin: Nyquist fix-up for bin 0 */

    uint32_t c_s = 0, c_par = 0, c_q = q0 + late * QB;
    for (uint32_t it = 0; it < n_iter; ++it)
    {
        if (late && (it == n_iter - 1))
            c_q             = q0;
        uint32_t rows   = min(QB, q1 - c_q);
        mbar_wait(&full[c_s], c_par);

        const float4 *g4 = reinterpret_cast<const float4 *>(sG + size_t(c_s) * stage_elems);
        const float4 *x4 = reinterpret_cast<const float4 *>(sX + size_t(c_s) * stage_elems);
        for (uint32_t r = 0; r < rows; ++r)
        {
            #pragma unroll
            for (int v = 0; v < MAC_VPT; ++v)
            {
                float4 g    = g4[r * (TB / 2) + tid + v * T];
                float4 x    = x4[r * (TB / 2) + tid + v * T];
                acc[v].x    = fmaf(g.x, x.x, acc[v].x);
                acc[v].y    = fmaf(g.x, x.y, acc[v].y);
                acc[v].z    = fmaf(g.z, x.z, acc[v].z);
                acc[v].w    = fmaf(g.z, x.w, acc[v].w);
                acc[v].x    = fmaf(-g.y, x.y, acc[v].x);
                acc[v].y    = fmaf(g.y, x.x, acc[v].y);
                acc[v].z    = fmaf(-g.w, x.w, acc[v].z);
                acc[v].w    = fmaf(g.w, x.z, acc[v].w);
                if (v == 0)
                    dny         = fmaf(g.y, x.y, dny);
            }
        }
        c_q            += QB;
        if (++c_s == NS)    { c_s = 0; c_par ^= 1u; }

        __syncthreads();            /* everyone is done with that stage: refill it */
        if ((tid == 0) && (f_it < n_iter))
            issue_next();
    }

    /* bin 0 holds (DC, Nyquist): both real, multiplied separately.  The complex MAC above gave
     * x = sum(re*re - im*im), so re = x + sum(im*im), im = sum(im*im). */
    if ((tile == 0) && (tid == 0))
    {
        acc[0].x   += dny;
        acc[0].y    = dny;
    }

    /* launched early: the previous launch may still be reading the rows this one replaces
     * (STEP_AHEAD: it cannot -- the rows have a slot of their own, free once chain_head says so) */
    CHAIN_STAMP(blockIdx.x + gridDim.x * blockIdx.y, 1);
    const bool ahead = (a.flags & STEP_AHEAD) != 0;
    if (!ahead)
        asm volatile("griddepcontrol.wait;" ::: "memory");
    CHAIN_STAMP(blockIdx.x + gridDim.x * blockIdx.y, 2);
    if ((!ahead) && (a.chain_head != nullptr) && (blockIdx.x == 0) && (blockIdx.y == 0) && (tid == 0))
        asm volatile("st.release.gpu.global.u32 [%0], %1;" :: "l"(a.chain_head), "r"(uint32_t(a.t_base + a.frame0) + 1u) : "memory");

    float4 *yp      = reinterpret_cast<float4 *>(a.ypart + (uint64_t(jobi) * rows_per_job(a) + a.row0 + split) * M
                                                 + uint64_t(tile) * TB);
    #pragma unroll
    for (int v = 0; v < MAC_VPT; ++v)
        yp[tid + v * T] = acc[v];

    if (a.fold_tickets != nullptr)
        fold_rows(a.fold_tickets + jobi, a.ypart + (uint64_t(jobi) * rows_per_job(a) + a.row0) * M, a.splits,
                  a.splits * gridDim.y, M, tid, T);
    /* STEP_AHEAD: this launch completes after every launch before it (stream order for what follows) */
    if (ahead && (blockIdx.x == 0) && (blockIdx.y == 0) && (tid == 0))
        asm volatile("griddepcontrol.wait;" ::: "memory");
}

/* ------------------------------------------------------------------------------------------- */
/* k_mac_multi<TF> : TF consecutive frames of every instance in ONE pass over the IR spectra      */
/* (calls that bring several whole frames: offline rendering, BASELINE config 4).                */
/*                                                                                             */
/*   Y_{t+j}[k] = sum_q G_q[k] X_{t+j-q}[k],  j = 0 .. TF-1                                       */
/*                                                                                             */
/* For a fixed q the TF frames need the ring rows X_{t-q} .. X_{t-q+TF-1}; stepping q -> q+1      */
/* slides that window by one row.  Every thread keeps the window for its bins in registers        */
/* (a rotating register file, statically indexed: the step loop is dispatched on step % TF), so a */
/* step still loads just one IR row and ONE ring row from shared memory -- the HBM bytes per      */
/* output sample drop by TF, the shared-memory traffic per step does not grow.                    */
/* Partial rows go to ypart[(j * n_active + job) * splits + split], the order k_inv expects for   */
/* a launch over TF * n_active frame-jobs.                                                       */

template <int TF, int PH>
__device__ __forceinline__ void multi_step(float4 (&acc)[TF], float4 (&win)[TF], float (&dny)[TF],
                                           const float4 *g4, const float4 *x4, uint32_t col, bool fix0)
{
    /* the row that enters the window at this step is frame 0's operand */
    constexpr int NEW = (TF - PH) % TF;
    const float4 g  = g4[col];
    win[NEW]        = x4[col];
    #pragma unroll
    for (int j = 0; j < TF; ++j)
    {
        const float4 x  = win[(j + TF - PH) % TF];
        acc[j].x        = fmaf(g.x, x.x, acc[j].x);
        acc[j].y        = fmaf(g.x, x.y, acc[j].y);
        acc[j].z        = fmaf(g.z, x.z, acc[j].z);
        acc[j].w        = fmaf(g.z, x.w, acc[j].w);
        acc[j].x        = fmaf(-g.y, x.y, acc[j].x);
        acc[j].y        = fmaf(g.y, x.x, acc[j].y);
        acc[j].z        = fmaf(-g.w, x.w, acc[j].z);
        acc[j].w        = fmaf(g.w, x.z, acc[j].w);
    }
    /* Nyquist fix-up of packed bin 0: only the warp that owns column 0 needs it */
    if (fix0)
    {
        #pragma unroll
        for (int j = 0; j < TF; ++j)
            dny[j]          = fmaf(g.y, win[(j + TF - PH) % TF].y, dny[j]);
    }
}

__device__ __forceinline__ void mbar_arrive(uint64_t *bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(smem_u32(bar)) : "memory");
}

/* blockDim.x = TB/2 consumer threads (one float4 column = 2 bins each) + one producer warp.
 * The register window limits occupancy to one CTA per SM at TF = 8, so latency is hidden inside
 * the CTA instead: a dedicated producer warp keeps an NS-deep TMA ring full, consumers hand
 * stages back through per-stage "empty" mbarriers, and there is no CTA-wide barrier in the loop. */
template <int TF>
__global__ void __launch_bounds__(544)
k_mac_multi(const StepArgs a, const MacShape sh)
{
    static_assert((TF == 2) || (TF == 4) || (TF == 8), "k_mac_multi: TF must be 2, 4 or 8");
    extern __shared__ __align__(128) unsigned char smraw[];

    const uint32_t M        = 1u << (a.rank - 1);
    const uint32_t TB       = sh.TB, QB = sh.QB, NS = sh.NS;
    const uint32_t CONS     = blockDim.x - 32;              /* consumer threads = TB / 2 */
    const uint32_t tid      = threadIdx.x;
    const uint32_t jobi     = blockIdx.x / a.splits;        /* = index into the active list */
    const uint32_t split    = blockIdx.x % a.splits;
    const uint32_t tile     = blockIdx.y;

    const uint32_t stage_elems = QB * TB;
    float2 *sG              = reinterpret_cast<float2 *>(smraw);
    float2 *sX              = sG + size_t(NS) * stage_elems;
    uint64_t *full          = reinterpret_cast<uint64_t *>(sX + size_t(NS) * stage_elems);
    uint64_t *empty         = full + NS;

    /* job of the FIRST frame of the group: slot0 = ring slot of X_t */
    const Job job           = fetch_job(a, jobi);
    const InstDesc d        = a.inst[job.inst];

    uint32_t qa             = max(job.qa, d.q_lo);
    uint32_t qb             = min(job.qb, d.q_lo + d.nq);
    uint32_t nq             = (qb > qa) ? (qb - qa) : 0;
    uint32_t c0, c1;
    chunk_range(nq, split, a.splits, 0, c0, c1);
    const uint32_t q0       = qa + c0, q1 = qa + c1;
    const uint32_t n_iter   = (q1 - q0 + QB - 1) / QB;

    const float2 *Gt        = d.G + uint64_t(tile) * TB;
    const float2 *Xt        = d.ring + uint64_t(tile) * TB;
    const uint32_t row_bytes = TB * uint32_t(sizeof(float2));
    const uint64_t l2_stream = stream_policy();

    if (tid == 0)
    {
        for (uint32_t s = 0; s < NS; ++s)
        {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], CONS / 32);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    __syncthreads();

    if (tid >= CONS)
    {
        /* ---- producer warp: one lane feeds the ring ---- */
        if (tid == CONS)
        {
            uint32_t f_s = 0, f_par = 1, f_q = q0;
            uint32_t f_slot = uint32_t((uint64_t(job.slot0) + q0) % d.S);
            for (uint32_t it = 0; it < n_iter; ++it)
            {
                if (it >= NS)
                    mbar_wait(&empty[f_s], f_par);                  /* consumers released use it - NS */
                uint32_t rows   = min(QB, q1 - f_q);
                float2 *g       = sG + size_t(f_s) * stage_elems;
                float2 *x       = sX + size_t(f_s) * stage_elems;
                mbar_expect_tx(&full[f_s], 2u * rows * row_bytes);
                bulk_g2s(g, Gt + uint64_t(f_q - d.q_lo) * M, rows * row_bytes, &full[f_s], l2_stream);
                uint32_t n1     = min(rows, d.S - f_slot);
                bulk_g2s(x, Xt + uint64_t(f_slot) * M, n1 * row_bytes, &full[f_s], l2_stream);
                if (n1 < rows)
                    bulk_g2s(x + size_t(n1) * TB, Xt, (rows - n1) * row_bytes, &full[f_s], l2_stream);
                f_q            += QB;
                f_slot         += QB;
                if (f_slot >= d.S)  f_slot -= d.S;
                if (++f_s == NS)    { f_s = 0; f_par ^= 1u; }       /* parity of use (it/NS - 1) */
            }
        }
        return;
    }

    /* ---- consumers ---- */
    float4 acc[TF], win[TF];
    float dny[TF];
    #pragma unroll
    for (int j = 0; j < TF; ++j)
    {
        dny[j]          = 0.0f;
        acc[j]          = win[j] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    }

    /* window rows of the later frames at the first step: frame j needs X_{t+j-q0}, which sits
     * j slots BEFORE the slot of X_{t-q0} (newer frames live in lower slots) */
    if (n_iter > 0)
    {
        #pragma unroll
        for (int j = 1; j < TF; ++j)
        {
            uint32_t slot   = uint32_t((uint64_t(job.slot0) + q0 + uint64_t(d.S) * TF - uint32_t(j)) % d.S);
            win[j]          = __ldg(reinterpret_cast<const float4 *>(Xt + uint64_t(slot) * M) + tid);
        }
    }

    const bool fix0 = (tile == 0) && (tid < 32);        /* warp-uniform */
    uint32_t step = 0, c_s = 0, c_par = 0, c_q = q0;
    for (uint32_t it = 0; it < n_iter; ++it)
    {
        const uint32_t s = c_s;
        uint32_t rows   = min(QB, q1 - c_q);
        mbar_wait(&full[s], c_par);

        const float4 *g4 = reinterpret_cast<const float4 *>(sG + size_t(s) * stage_elems);
        const float4 *x4 = reinterpret_cast<const float4 *>(sX + size_t(s) * stage_elems);
        for (uint32_t r = 0; r < rows; ++r, ++step)
        {
            const float4 *gr = g4 + r * (TB / 2), *xr = x4 + r * (TB / 2);
            switch (step & (TF - 1))
            {
                case 0: multi_step<TF, 0>(acc, win, dny, gr, xr, tid, fix0); break;
                case 1: multi_step<TF, 1 % TF>(acc, win, dny, gr, xr, tid, fix0); break;
                case 2: multi_step<TF, 2 % TF>(acc, win, dny, gr, xr, tid, fix0); break;
                case 3: multi_step<TF, 3 % TF>(acc, win, dny, gr, xr, tid, fix0); break;
                case 4: multi_step<TF, 4 % TF>(acc, win, dny, gr, xr, tid, fix0); break;
                case 5: multi_step<TF, 5 % TF>(acc, win, dny, gr, xr, tid, fix0); break;
                case 6: multi_step<TF, 6 % TF>(acc, win, dny, gr, xr, tid, fix0); break;
                default: multi_step<TF, 7 % TF>(acc, win, dny, gr, xr, tid, fix0); break;
            }
        }

        c_q            += QB;
        if (++c_s == NS)    { c_s = 0; c_par ^= 1u; }

        /* this warp is done with stage s */
        __syncwarp();
        if ((tid & 31) == 0)
            mbar_arrive(&empty[s]);
    }

    #pragma unroll
    for (int j = 0; j < TF; ++j)
    {
        if ((tile == 0) && (tid == 0))
        {
            acc[j].x       += dny[j];
            acc[j].y        = dny[j];
        }
        float4 *yp      = reinterpret_cast<float4 *>(
            a.ypart + ((uint64_t(j) * a.n_active + jobi) * a.splits + split) * M + uint64_t(tile) * TB);
        yp[tid]         = acc[j];
    }
}

/* ------------------------------------------------------------------------------------------- */
/* partial_outputs : the samples of the frame in progress against taps [0, F) in direct form       */
/* (reference: dsp::convolve and the raising levels, Convolver.cpp:251-262,295) -- zero latency    */
/* for any call size:                                                                           */
/*     dst[i] = pend[off + i] + sum_{j <= off + i} cur[j] * head[off + i - j],   i in [i0, i1)     */
/* Parallel across outputs AND taps: a group of G lanes (a power of two, inside one warp) shares    */
/* one output, lane l takes the taps j = l, l + G, ... .  The taps are walked in tiles of PO_TILE:   */
/* the CTA stages cur[tile] and the matching window of `head` in shared memory with coalesced       */
/* loads (all in flight at once -- a serial chain of dependent global loads per tap is what made     */
/* the first version latency-bound), then every group sums its output's share of the tile from      */
/* shared memory: fp32 products in four independent chains, chain totals added in fp64 per tile,     */
/* group totals by shuffle.  Samples newer than the group's newest output are never read (`cur`      */
/* beyond them is stale), taps beyond an output's own index meet a zero in the head window.          */
/* Every thread of the CTA must call it (T a multiple of 32, T <= PO_MAXT).                          */

/* asynchronous global -> shared copies of single words (no register, no stall at the copy) */
__device__ __forceinline__ void cp_async4(void *smem, const void *gmem)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" :: "r"(uint32_t(__cvta_generic_to_shared(smem))), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async8(void *smem, const void *gmem)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" :: "r"(uint32_t(__cvta_generic_to_shared(smem))), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all()
{
    asm volatile("cp.async.wait_all;" ::: "memory");
}

constexpr uint32_t PO_TILE  = 2048;
constexpr uint32_t PO_MAXT  = 512;
constexpr uint32_t PO_SMEM_FLOATS = 2 * PO_TILE + PO_MAXT;     /* cur tile | head window */

/* xnew != NULL: the samples j >= off are taken from xnew[j - off] (the caller's block) instead of   */
/* cur -- for CTAs that must not depend on another CTA's copy into `cur`; pend == NULL: the direct   */
/* sum alone (the pending block is added later, by whoever produces it).                             */
__device__ __forceinline__ void partial_outputs(const float *cur, const float *head, const float *pend,
                                                float *dst, uint32_t off, uint32_t i0, uint32_t i1,
                                                uint32_t tid, uint32_t T, float *po_smem,
                                                const float *xnew = nullptr)
{
    const uint32_t n        = i1 - i0;
    if (n == 0)
        return;
    uint32_t G              = 1;
    while ((G < 32) && (n * G * 2 <= T))
        G                     <<= 1;
    const uint32_t per_pass = T / G;                                /* outputs per window */
    const uint32_t lane     = tid % G, grp = tid / G;
    float *cs               = po_smem;                              /* cs[j - j0]                      */
    float *hs               = po_smem + PO_TILE;                    /* hs[k] = head[hbase + k]          */

    for (uint32_t base = 0; base < n; base += per_pass)            /* uniform trip counts throughout */
    {
        const uint32_t ia       = i0 + base;                        /* window of outputs [ia, ib) */
        const uint32_t ib       = min(ia + per_pass, i1);
        const uint32_t i        = ia + grp;
        const bool live         = i < ib;
        const uint32_t m_max    = off + ib - 1;                     /* newest sample of the window */
        double total            = 0.0;
        for (uint32_t j0 = 0; j0 <= m_max; j0 += PO_TILE)
        {
            /* head indices needed: (off + i) - j for i in [ia, ib), j in [j0, j0 + TILE) */
            const int32_t hbase     = int32_t(off + ia) - int32_t(j0) - int32_t(PO_TILE) + 1;
            const uint32_t hcount   = PO_TILE + (ib - ia) - 1;
            /* taps of this tile that exist: [j0, j0 + kend), kend a multiple of the 4 G stride */
            const uint32_t kend     = min(PO_TILE, (m_max - j0 + 4 * G) & ~(4 * G - 1));
            __syncthreads();                                        /* previous tile / window consumed */
            /* asynchronous copies: every word of the tile is in flight at once (plain loads into
             * shared memory were issued one round trip after the other) */
            for (uint32_t k = tid; k < kend; k += T)
            {
                const uint32_t j        = j0 + k;
                if (j > m_max)
                    cs[k]                   = 0.0f;
                else
                    cp_async4(cs + k, ((xnew != nullptr) && (j >= off)) ? (xnew + (j - off)) : (cur + j));
            }
            for (uint32_t k = (PO_TILE - kend) + tid; k < hcount; k += T)
            {
                const int32_t h         = hbase + int32_t(k);
                if (h >= 0)
                    cp_async4(hs + k, head + h);
                else
                    hs[k]                   = 0.0f;
            }
            cp_async_wait_all();
            __syncthreads();
            if (live)
            {
                /* head[(off + i) - j] = hs[(i - ia) + (TILE - 1) - (j - j0)] */
                const float *hp         = hs + (i - ia) + (PO_TILE - 1);
                float p0 = 0.0f, p1 = 0.0f, p2 = 0.0f, p3 = 0.0f;
                #pragma unroll 2
                for (uint32_t k = lane; k < kend; k += 4 * G)
                {
                    p0                      = fmaf(cs[k],         hp[-int32_t(k)],         p0);
                    p1                      = fmaf(cs[k + G],     hp[-int32_t(k + G)],     p1);
                    p2                      = fmaf(cs[k + 2 * G], hp[-int32_t(k + 2 * G)], p2);
                    p3                      = fmaf(cs[k + 3 * G], hp[-int32_t(k + 3 * G)], p3);
                }
                total                  += double((p0 + p1) + (p2 + p3));
            }
        }
        for (uint32_t sft = G >> 1; sft > 0; sft >>= 1)
            total                  += __shfl_xor_sync(0xffffffffu, total, sft);
        if (live && (lane == 0))
            dst[i]                  = ((pend != nullptr) ? pend[off + i] : 0.0f) + float(total);
    }
}

/* ------------------------------------------------------------------------------------------- */
/* k_frame : ranks 8..13, whole frames for every instance -- the block scheduler's "one launch    */
/* per block".  grid = (jobs * splits, M / TB), TB / 4 threads.                                   */
/*                                                                                             */
/*   every CTA            : streams its partition chunk exactly like k_mac and writes one        */
/*                          partial row; the CTAs of split 0 take the stage with partition q = 0  */
/*                          (the only one that needs the arriving frame's own spectrum) LAST;     */
/*   (split 0, tile 0)    : before that last stage it transforms the input frame (fwd_body) into  */
/*                          the ring and publishes it through ring_head;                         */
/*   the last CTA to      : (atomic ticket per job) sums the partial rows out of L2 and runs the  */
/*   finish a job           inverse transform (inv_body) -> output block (or the cross-GPU sum).  */
/*                                                                                             */
/* Launched with programmatic stream serialisation: the partition stream of block t+1 overlaps   */
/* the inverse-transform tail of block t.  Before griddepcontrol.wait a CTA touches only the IR   */
/* spectra (immutable between inits), ring rows announced through ring_head (acquire / release)   */
/* and tables written by stream-ordered copies.  The caller's INPUT block, the ring slot of the   */
/* arriving frame, the partial rows, the tickets and the output block are all touched AFTER       */
/* griddepcontrol.wait, i.e. when every earlier launch in the stream has completed and flushed -- */
/* so a src that an earlier launch produced (two batches cascaded on one stream, or a batch fed   */
/* its own dst) is final when it is read, whoever that producer was.                             */

/* acc += g * x for two packed complex bins; dn += Im g * Im x (the bin-0 Nyquist fix-up) */
__device__ __forceinline__ void cmac(float4 &acc, float &dn, const float4 g, const float4 x)
{
    acc.x           = fmaf(g.x, x.x, acc.x);
    acc.y           = fmaf(g.x, x.y, acc.y);
    acc.z           = fmaf(g.z, x.z, acc.z);
    acc.w           = fmaf(g.z, x.w, acc.w);
    acc.x           = fmaf(-g.y, x.y, acc.x);
    acc.y           = fmaf(g.y, x.x, acc.y);
    acc.z           = fmaf(-g.w, x.w, acc.z);
    acc.w           = fmaf(g.w, x.z, acc.w);
    dn              = fmaf(g.y, x.y, dn);
}

template <int RANK>
struct FrameCfg
{
    static constexpr int M      = 1 << (RANK - 1);
    static constexpr int TB     = (M < 1024) ? M : 1024;            /* bins per CTA tile       */
    static constexpr int T      = TB / 4;                           /* threads per CTA         */
    static constexpr int MINB   = (RANK >= 13) ? 2 : ((T >= 256) ? 4 : 8);  /* CTAs per SM (register cap) */
};

/* GEN = the job-list form for the general path: per job any of P1 / FFT / MAC + inverse / P2 (see
 * Job).  Every CTA waits for all earlier launches right after its prologue (griddepcontrol.wait),
 * so ring_head only orders CTAs of this launch. */
template <int RANK, bool GEN>
__device__ __forceinline__ void frame_body(const StepArgs &a, const MacShape &sh, uint32_t *tickets,
                                           const ReduceArgs &ra, const Job *pack)
{
    using C = FftCfg<RANK, FrameCfg<RANK>::T>;
    constexpr uint32_t M = C::M, T = C::T, TB = FrameCfg<RANK>::TB;
    static_assert(C::NH == 2, "k_frame: both FFT halves resident");
    static_assert(RANK <= 13, "k_frame: the frame transform must fit the stage buffers");

    extern __shared__ __align__(128) unsigned char smraw[];

    const uint32_t QB       = sh.QB, NS = sh.NS;
    const uint32_t tid      = threadIdx.x;
    const uint32_t jobi     = blockIdx.x / a.splits;
    const uint32_t split    = blockIdx.x % a.splits;
    const uint32_t tile     = blockIdx.y;

    /* stage s = [ G rows : stage_elems float2 | ring rows : stage_elems float2 ], back to back */
    const uint32_t stage_elems = QB * TB;                           /* 1024 float2 */
    float2 *stages          = reinterpret_cast<float2 *>(smraw);
    uint64_t *full          = reinterpret_cast<uint64_t *>(stages + size_t(NS) * 2 * stage_elems);
    uint32_t *flag          = reinterpret_cast<uint32_t *>(full + NS);

    /* let the next block's launch become resident as soon as this one frees SM slots */
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    FRAME_STAMP(0);
    if (tid == 0)
    {
        for (uint32_t s = 0; s < NS; ++s)
            mbar_init(&full[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    __syncthreads();

    /* the instance / job tables are written by stream-ordered memcpys, never by a kernel */
    const Job job           = (GEN && (a.jobs == nullptr)) ? pack[jobi] : fetch_job(a, jobi);
    const InstDesc d        = a.inst[job.inst];
    const bool split0       = (split == 0);
    const bool fft_cta      = split0 && (tile == 0);
    if (GEN && (!(job.flags & JOB_MAC)) && (!fft_cta))
        return;                                 /* a job without a partition sum needs one CTA */
    /* The job-list form touches per-instance state that the launch before it writes (the frame in
     * progress, the pending block, ring rows without a ring_head hand-shake across launches): it
     * orders itself behind every earlier launch HERE -- launched with programmatic serialisation
     * it has become resident, set up its barriers and fetched its job under the predecessor's tail. */
    if (GEN)
        asm volatile("griddepcontrol.wait;" ::: "memory");

    uint32_t qa             = max(job.qa, d.q_lo);
    uint32_t qb             = min(job.qb, d.q_lo + d.nq);
    /* lookahead (LA_BUFS): this launch streams bin slice la_c of the tails [qs, qb) of the next
     * group's blocks; its own head is [qa, qs) when its T is complete, else every partition */
    const uint32_t LK       = GEN ? 0u : a.la_K;
    const uint32_t qs       = (LK != 0) ? max(qa, min(qb, 2u * LK)) : qb;
    const uint32_t qe       = qb;
    if ((LK != 0) && a.la_use)
        qb                      = qs;
    uint32_t nq             = ((qb > qa) && ((!GEN) || (job.flags & JOB_MAC))) ? (qb - qa) : 0;
    uint32_t c0, c1;
    chunk_range(nq, split, a.splits, sh.bias, c0, c1);
    const uint32_t q0       = qa + c0, q1 = qa + c1;
    const uint32_t n_iter   = (q1 - q0 + QB - 1) / QB;
    /* Split 0 owns the partitions that need the NEWEST spectra: q = 0 the arriving frame's own
     * (written by this launch), q = 1 the previous frame's (published near the END of the previous
     * launch's partition stream, and CTAs of this launch may have become resident long before
     * that).  The `late` stages holding them go last, newest last:
     *     stage order  late, late + 1, ..., n_iter - 1, late - 1, ..., 0.                        */
    const uint32_t late     = split0 ? min(n_iter, (QB == 1) ? 2u : 1u) : 0u;
    const uint32_t n_main   = split0 ? ((n_iter > 0) ? n_iter - 1 : 0) : n_iter;   /* all but stage 0 */

    const float2 *Gt        = d.G + uint64_t(tile) * TB;            /* row r at Gt + r * M */
    const float2 *Xt        = d.ring + uint64_t(tile) * TB;
    const uint32_t row_bytes = TB * uint32_t(sizeof(float2));

    /* Lookahead tail, as a "virtual row" of M bins: segment j (W = M / K bins) of the row of partition q
     * is  G_q[slice] * X_{t0 + K + j - q}[slice]  -- the same multiply-add as the head rows.  A tile of
     * TB virtual bins covers nj segments j0 .. j0 + nj - 1 (or a part of one: Wg bins at offset p0 of
     * the slice).  The CTA's partitions tq0 .. tq1 - 1 go QT per stage.  Its ring slices form ONE
     * window: slice s = 0 .. tq1 - tq0 + nj - 2 is frame t0 + K + j0 + nj - 1 - tq0 - s (ascending ring
     * slots), which segment j reads for partition tq0 + s - (nj - 1 - j).  Shared memory holds NS
     * buffers of QT G slices, then a circular window of NW = NS QT + nj - 1 slices (slice s in slot
     * s % NW).  Tail stage k copies its G slices and only the window slices k QT + nj - 1 ..
     * (k + 1) QT + nj - 2 (stage 0 also the first nj - 1): each ring slice is copied once.  Those
     * overwrite slices (k - NS) QT .., which stage k - NS was the last to read -- and stage k is issued
     * after every thread has passed stage k - NS. */
    uint32_t tq0 = 0, tq1 = 0, n_titer = 0, QT = 1, NW = 1, Wg = 0, Wc4 = 1, nj = 1, boff = 0, slot_w0 = 0;
    if (LK != 0)
    {
        const uint32_t W    = M / LK;
        Wg                  = min(W, TB);
        Wc4                 = Wg / 2;
        nj                  = max(1u, TB / W);
        const uint32_t j0   = (tile * TB) / W;
        boff                = a.la_c * W + (tile * TB) % W;                 /* bin offset of the slices */
        QT                  = ((2u * NS * stage_elems) / Wg - (nj - 1)) / (2u * NS);
        NW                  = NS * QT + nj - 1;
        uint32_t e0, e1;
        chunk_range(qe - qs, split, a.splits, sh.bias, e0, e1);
        tq0                 = qs + e0;
        tq1                 = qs + e1;
        n_titer             = (tq1 - tq0 + QT - 1) / QT;
        /* window slice s is frame fmax - s, fmax = t0 + K + j0 + nj - 1 - tq0, in ring slot
         * (slot0 + t - fmax + s) mod S (t - fmax >= 1 when the CTA has a tail) */
        if (n_titer > 0)
            slot_w0             = uint32_t((uint64_t(job.slot0) + (a.la_c + tq0 + 1u - (LK + j0 + nj))) % d.S);
    }
    const uint32_t t0       = job.tlo - a.la_c;                    /* first block of this launch's group */

    /* Stage-ring bookkeeping is incremental (next stage buffer, next ring slot): no integer
     * division inside the streaming loop.  `issued` = stages fetched so far. */
    const uint32_t slot_q0  = uint32_t((uint64_t(job.slot0) + q0) % d.S);
    uint32_t issued = 0, f_s = 0;
    uint32_t f_slot         = slot_q0 + late * QB;
    if (f_slot >= d.S)      f_slot -= d.S;
    uint32_t t_issued = 0;
    auto issue_next = [&]()                     /* thread 0 only */
    {
        if (t_issued < n_titer)
        {
            /* a lookahead tail stage: partitions q .. q + rows - 1 of bin slice la_c */
            const uint32_t q    = tq0 + t_issued * QT;
            const uint32_t rows = min(QT, tq1 - q);
            if (t_issued == 0)
            {
                /* the tails read frames <= t0 - 1 (the oldest one, t0 + K - (bins + 1) + 1, is newer than
                 * the oldest frame a launch without lookahead reads: the ring size is unchanged) */
                wait_ge<false>(a.ring_head + job.inst, t0, a.error, SPIN_ERR_RING);
                asm volatile("fence.proxy.async;" ::: "memory");
            }
            /* new window slices s0 .. s0 + nx - 1 */
            const uint32_t s0   = (t_issued == 0) ? 0u : t_issued * QT + nj - 1;
            const uint32_t nx   = rows + ((t_issued == 0) ? nj - 1 : 0u);
            const uint32_t sb   = Wg * uint32_t(sizeof(float2));
            float2 *g           = stages + size_t(f_s) * QT * Wg;
            float2 *xw          = stages + size_t(NS) * QT * Wg;
            mbar_expect_tx(&full[f_s], (rows + nx) * sb);
            for (uint32_t r = 0; r < rows; ++r)
                bulk_g2s(g + size_t(r) * Wg, d.G + uint64_t(q + r - d.q_lo) * M + boff, sb, &full[f_s], stream_policy());
            uint32_t ws         = s0 % NW;
            uint32_t sl         = (slot_w0 + s0) % d.S;
            for (uint32_t i = 0; i < nx; ++i)
            {
                bulk_g2s(xw + size_t(ws) * Wg, d.ring + uint64_t(sl) * M + boff, sb, &full[f_s], stream_policy());
                if (++ws == NW)     ws = 0;
                if (++sl == d.S)    sl = 0;
            }
            ++t_issued;
            if (++f_s == NS)    f_s = 0;
            return;
        }
        uint32_t stg;
        if (issued < n_iter - late)
        {
            stg             = late + issued;
            if (issued == 0)
            {
                /* partitions q >= q0 + late * QB need frames <= t - (q0 + late * QB) */
                wait_ge<false>(a.ring_head + job.inst, job.tlo - (q0 + late * QB) + 1u, a.error, SPIN_ERR_RING);
                asm volatile("fence.proxy.async;" ::: "memory");
            }
        }
        else
        {
            stg             = n_iter - 1 - issued;
            f_slot          = slot_q0 + stg * QB;
            if (f_slot >= d.S)  f_slot -= d.S;
            if (stg != 0)
            {
                /* the previous frame's spectrum: the previous launch publishes it late */
                wait_ge<false>(a.ring_head + job.inst, job.tlo - (q0 + stg * QB) + 1u, a.error, SPIN_ERR_RING);
                asm volatile("fence.proxy.async;" ::: "memory");
            }
        }
        uint32_t q      = q0 + stg * QB;
        uint32_t rows   = min(QB, q1 - q);
        float2 *g       = stages + size_t(f_s) * 2 * stage_elems;
        float2 *x       = g + stage_elems;
        /* (an L2 policy is one instruction: made here rather than held in registers across the loops)
         * the head rows of a lookahead launch are read again by the next 2K - 1 launches: keep them in L2 */
        const uint64_t l2_head = (LK != 0) ? keep_policy() : stream_policy();
        mbar_expect_tx(&full[f_s], 2u * rows * row_bytes);
        bulk_g2s(g, Gt + uint64_t(q - d.q_lo) * M, rows * row_bytes, &full[f_s], l2_head);
        uint32_t n1     = min(rows, d.S - f_slot);
        bulk_g2s(x, Xt + uint64_t(f_slot) * M, n1 * row_bytes, &full[f_s], l2_head);
        if (n1 < rows)
            bulk_g2s(x + size_t(n1) * TB, Xt, (rows - n1) * row_bytes, &full[f_s], l2_head);
        ++issued;
        if (++f_s == NS)    f_s = 0;
        f_slot         += QB;
        if (f_slot >= d.S)  f_slot -= d.S;
    };

    /* the head stages use the stage buffers that the tail's window covers: they follow the tail */
    if (tid == 0)
        while ((t_issued + issued < NS) && (t_issued + issued < ((n_titer > 0) ? n_titer : n_main)))
            issue_next();

    float *po               = nullptr;
    /* GEN: a job with a partition sum has splits x tiles CTAs of which all but one idle once their
     * chunk is streamed, while the direct-form answers (P1: the samples that continue the frame in
     * progress; P2: the first samples of the next frame) were the longest stretch of the one CTA
     * that also transforms.  So they are SPREAD: every other CTA of the job computes a slice of
     * both direct sums while its first stages are in flight (P1 complete, with the OLD pending
     * block; P2 without the new one) into the job's answer row behind the partial rows; the CTA
     * that finishes the job copies them out (adding the new pending block to P2) after the ticket,
     * i.e. after every CTA has read the caller's samples -- safe for in-place calls. */
    const uint32_t n_cta    = a.splits * gridDim.y;
    const bool spread       = GEN && ((job.flags & JOB_MAC) != 0) && (n_cta > 1);
    constexpr uint32_t AW   = TB;           /* floats per answer array in the scratch: a segment has <= min(F, 1024) samples */
    constexpr bool TW_FITS  = GEN && (3 * AW + 2 * uint32_t(C::TW_TOTAL) <= PO_SMEM_FLOATS);   /* ranks 8..10 */
    const bool tw_early     = TW_FITS && fft_cta && (spread || ((job.n == 0) && (job.n2 == 0)));
    float *ans1             = nullptr, *ans2 = nullptr;
    if constexpr (GEN)
    {
        __shared__ __align__(16) float po_scratch[PO_SMEM_FLOATS];
        po                      = po_scratch;
        if (spread)
        {
            ans1                    = reinterpret_cast<float *>(a.ypart + (uint64_t(a.n_jobs) * rows_per_job(a) + jobi) * M);
            ans2                    = ans1 + M;
        }
        if (tw_early)
        {
            /* this CTA's direct-form scratch is idle: the twiddles of its two transforms arrive
             * there while the partition stream runs, instead of at the head of each transform */
            float2 *tws             = reinterpret_cast<float2 *>(po + 3 * AW);
            for (uint32_t i = tid; i < uint32_t(C::TW_TOTAL); i += T)
                cp_async8(tws + i, a.tw + i);
        }
        if (fft_cta && (job.n > 0))
        {
            /* P1: the call's samples that continue the frame in progress, answered at once (from
             * the OLD pending block) while the first partition stages are in flight */
            for (uint32_t i = tid; i < job.n; i += T)
                d.cur[job.off + i]  = job.psrc[i];
            __syncthreads();                    /* the transform below reads them back */
            if (!spread)
            {
                partial_outputs(d.cur, d.head, d.pend, job.pdst, job.off, 0, job.n, tid, T, po);
                __syncthreads();
            }
        }
        if (spread && (!fft_cta))
        {
            /* a page-locked HOST block: every helper fetches the samples its slice needs across PCIe,
             * so fewer, larger slices */
            const uint32_t ci       = split * gridDim.y + tile - 1u;
            const uint32_t nc       = (a.flags & STEP_HOST_IO) ? min(n_cta - 1u, 8u) : (n_cta - 1u);
            if ((job.n > 0) && (ci < nc))
                partial_outputs(d.cur, d.head, d.pend, ans1, job.off,
                                uint32_t((uint64_t(job.n) * ci) / nc), uint32_t((uint64_t(job.n) * (ci + 1)) / nc),
                                tid, T, po, job.psrc);
            if ((job.n2 > 0) && (ci < nc))
            {
                __syncthreads();
                partial_outputs(d.cur, d.head, nullptr, ans2, job.off2,
                                uint32_t((uint64_t(job.n2) * ci) / nc), uint32_t((uint64_t(job.n2) * (ci + 1)) / nc),
                                tid, T, po, job.psrc2);
            }
        }
        FRAME_STAMP(4);
    }

    float4 acc[MAC_VPT];
    #pragma unroll
    for (int v = 0; v < MAC_VPT; ++v)
        acc[v]      = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    float dny       = 0.0f;

    uint32_t c_s = 0, c_par = 0, c_n = 0;
    auto consume = [&]()
    {
        const uint32_t stg = (c_n < n_iter - late) ? (late + c_n) : (n_iter - 1 - c_n);
        uint32_t rows   = min(QB, q1 - (q0 + stg * QB));
        mbar_wait(&full[c_s], c_par);

        const float4 *g4 = reinterpret_cast<const float4 *>(stages + size_t(c_s) * 2 * stage_elems);
        const float4 *x4 = g4 + stage_elems / 2;
        for (uint32_t r = 0; r < rows; ++r)
        {
            #pragma unroll
            for (int v = 0; v < MAC_VPT; ++v)
            {
                float4 g    = g4[r * (TB / 2) + tid + v * T];
                float4 x    = x4[r * (TB / 2) + tid + v * T];
                acc[v].x    = fmaf(g.x, x.x, acc[v].x);
                acc[v].y    = fmaf(g.x, x.y, acc[v].y);
                acc[v].z    = fmaf(g.z, x.z, acc[v].z);
                acc[v].w    = fmaf(g.z, x.w, acc[v].w);
                acc[v].x    = fmaf(-g.y, x.y, acc[v].x);
                acc[v].y    = fmaf(g.y, x.x, acc[v].y);
                acc[v].z    = fmaf(-g.w, x.w, acc[v].z);
                acc[v].w    = fmaf(g.w, x.z, acc[v].w);
                if (v == 0)
                    dny         = fmaf(g.y, x.y, dny);
            }
        }
        ++c_n;
        if (++c_s == NS)        { c_s = 0; c_par ^= 1u; }
    };

    if (LK != 0)
    {
        /* The lookahead tail.  With several segments per tile (nj >= 2) a thread owns one float4 column
         * and the two segments jv, jv + 1: segment jv + 1 multiplies partition q by the window slice that
         * segment jv multiplied partition q - 1 by, so it comes from a register, and a partition costs the
         * thread one G and one X load for both.  A tile inside one segment (nj = 1): columns tid and
         * tid + T.  Every output still sums its partitions in ascending order, one fmaf chain each. */
        const bool run      = (nj > 1);
        const uint32_t col  = run ? tid % Wc4 : tid;
        const uint32_t jv0  = run ? 2u * (tid / Wc4) : 0u;
        float tdn[MAC_VPT]  = { 0.0f, 0.0f };
        auto tail = [&](auto run_c)
        {
            constexpr bool RUN  = decltype(run_c)::value;
            uint32_t xs         = nj - 1 - jv0;     /* window slot of segment jv0's operand for the next partition */
            float4 xp           = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
            const float4 *xw    = reinterpret_cast<const float4 *>(stages + size_t(NS) * QT * Wg);
            for (uint32_t it = 0; it < n_titer; ++it)
            {
                const uint32_t rows = min(QT, tq1 - (tq0 + it * QT));
                mbar_wait(&full[c_s], c_par);
                const float4 *g4 = reinterpret_cast<const float4 *>(stages + size_t(c_s) * QT * Wg);
                if (RUN && (it == 0))
                    xp              = xw[(xs - 1) * Wc4 + col];
                #pragma unroll 2
                for (uint32_t r = 0; r < rows; ++r)
                {
                    const float4 g  = g4[r * Wc4 + col];
                    const float4 x  = xw[xs * Wc4 + col];
                    cmac(acc[0], tdn[0], g, x);
                    if constexpr (RUN)
                    {
                        cmac(acc[1], tdn[1], g, xp);
                        xp              = x;
                    }
                    else
                        cmac(acc[1], tdn[1], g4[r * Wc4 + col + T], xw[xs * Wc4 + col + T]);
                    if (++xs == NW) xs = 0;
                }
                if (++c_s == NS)    { c_s = 0; c_par ^= 1u; }
                __syncthreads();
                if ((tid == 0) && (t_issued < n_titer))
                    issue_next();
            }
        };
        if (run)
            tail(std::true_type());
        else
            tail(std::false_type());
        /* every thread is past the last tail stage: the head stages may take the stage buffers */
        if (tid == 0)
            while ((issued < NS) && (issued < n_main))
                issue_next();
        FRAME_STAMP(4);
        /* bin 0 (DC, Nyquist) of the spectrum opens slice 0 of every segment */
        #pragma unroll
        for (int v = 0; v < MAC_VPT; ++v)
            if ((boff == 0) && (col + (run ? 0u : v * T) == 0))
            {
                acc[v].x       += tdn[v];
                acc[v].y        = tdn[v];
            }
        /* buffer la_put was last read by the blocks of the group LA_BUFS - 1 before the next one */
        if (tid == 0)
            wait_ge<false>(a.la_cons + size_t(a.la_put) * a.n_cap + job.inst, a.la_put_need, a.error, SPIN_ERR_RING);
        __syncthreads();
        float2 *tb      = a.la_T + uint64_t(a.la_put) * a.n_jobs * LK * a.splits * M + boff;
        #pragma unroll
        for (int v = 0; v < MAC_VPT; ++v)
        {
            const uint32_t j    = (tile * TB) / (M / LK) + jv0 + (run ? v : 0u);
            float4 *tp          = reinterpret_cast<float4 *>(tb + ((uint64_t(jobi) * LK + j) * a.splits + split) * M)
                                  + col + (run ? 0u : v * T);
            __stcg(tp, acc[v]);
            acc[v]              = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        }
        __threadfence();
        __syncthreads();
        if (tid == 0)
            asm volatile("red.release.gpu.global.add.u32 [%0], 1;"
                         :: "l"(a.la_prod + size_t(a.la_put) * a.n_cap + job.inst) : "memory");
        FRAME_STAMP(5);
    }

    for (uint32_t it = 0; it < n_main; ++it)
    {
        consume();
        __syncthreads();
        if ((tid == 0) && (issued < n_main))
            issue_next();
    }

    if (GEN)
        FRAME_STAMP(5);
    else if (LK != 0)
        FRAME_STAMP(6);
    if (split0)
    {
        if (fft_cta)
        {
            /* The input block is the caller's: an earlier launch in the stream may have produced
             * it (and that launch may still be in its tail while this one streams), so it is read
             * only once every earlier launch has completed.  That also retires every reader of
             * ring slot (-t) mod S.  Exception: the host knows the predecessor (STEP_EARLY_SRC). */
            if (!(a.flags & STEP_EARLY_SRC))
                asm volatile("griddepcontrol.wait;" ::: "memory");
            if ((!GEN) || (job.flags & JOB_FFT))
            {
            /* every stage buffer is idle here: two work buffers (one at rank 13) + the twiddle table */
            constexpr bool FFT_PP       = (RANK <= 12);
            constexpr uint32_t FFT_WORK = C::WORK * (FFT_PP ? 2 : 1);
            float2 *wa          = stages, *wb = FFT_PP ? stages + C::WORK : nullptr;
            const float2 *tw    = a.tw;
            if (tw_early)
            {
                cp_async_wait_all();
                tw                  = reinterpret_cast<const float2 *>(po + 3 * AW);    /* visible after fwd_body's first barrier */
            }
            else if (FFT_WORK + uint32_t(C::TW_TOTAL) <= NS * 2 * stage_elems)
            {
                float2 *tws         = stages + FFT_WORK;
                for (uint32_t i = tid; i < uint32_t(C::TW_TOTAL); i += T)
                    tws[i]              = a.tw[i];
                tw                  = tws;          /* visible after fwd_body's first barrier */
            }
            fwd_body<RANK, FFT_PP, int(T)>(wa, wb, job.src, job.spec, a.tw, tw, int(tid));
            /* generic-proxy global writes -> visible to the TMA (async proxy) reads issued below;
             * the same fence orders the scratch use of the stage buffers before their refill */
            __threadfence();
            asm volatile("fence.proxy.async;" ::: "memory");
            __syncthreads();
            if (tid == 0)
            {
                /* Publish "frames 0 .. t are in the ring" -- strictly in frame order (the
                 * acquire / release chain makes every older spectrum visible to whoever acquires
                 * the new value). */
                uint32_t *hp    = a.ring_head + job.inst;
                if (!GEN)
                    wait_ge<false>(hp, job.tlo, a.error, SPIN_ERR_RING);
                const uint32_t head = (GEN && (job.flags & JOB_FFT_PREV)) ? job.tlo : job.tlo + 1u;
                asm volatile("st.release.gpu.global.u32 [%0], %1;" :: "l"(hp), "r"(head) : "memory");
            }
            }
            if (GEN)
                FRAME_STAMP(6);
            if (GEN && (!(job.flags & JOB_MAC)))
                return;
        }
        else if ((tid == 0) && (n_iter > 0))
        {
            /* the other bin tiles of split 0 (ranks 12 / 13) learn through ring_head that the
             * arriving frame's spectrum has landed */
            wait_ge<false>(a.ring_head + job.inst, job.tlo - q0 + 1u, a.error, SPIN_ERR_RING);
        }
        if (n_iter > 0)
        {
            if (tid == 0)
            {
                asm volatile("fence.proxy.async;" ::: "memory");
                issue_next();
            }
            consume();
        }
    }

    if ((tile == 0) && (tid == 0))
    {
        acc[0].x   += dny;
        acc[0].y    = dny;
    }
    FRAME_STAMP(1);

    const bool pipelined    = (!GEN) && (a.slot_done != nullptr);
    uint32_t *my_done       = pipelined ? a.slot_done + size_t(a.seq % uint32_t(FRAME_SLOTS)) * a.n_cap + job.inst : nullptr;
    if (pipelined)
    {
        /* the slot (partial rows, tickets) was last used by launch seq - FRAME_SLOTS: its tail for
         * this instance must have finished (see FRAME_SLOTS) */
        if (tid == 0)
            wait_ge<false>(my_done, a.seq + 1u - uint32_t(FRAME_SLOTS), a.error, SPIN_ERR_RING);
        __syncthreads();
    }
    if ((!pipelined) || (a.flags & (STEP_HEAD_ONLY | STEP_ORDER_DST)))
    {
        /* not pipelined: partial rows, tickets and the output block are shared with the previous
         * launch's tail.  STEP_HEAD_ONLY: the other rows of this job come from the pending MAC launched
         * right before -- a true dependency on that launch's completion.  STEP_ORDER_DST: the output
         * block is still in use by a launch in flight. */
        asm volatile("griddepcontrol.wait;" ::: "memory");
    }

    const uint32_t rows = rows_per_job(a);
    float2 *yrow    = a.ypart + uint64_t(jobi) * rows * M;
    const float2 *ysum  = yrow + uint64_t(a.sum0) * M;              /* the rows the inverse transform adds */
    const uint32_t nsum = rows - a.sum0;
    float4 *yp      = reinterpret_cast<float4 *>(yrow + uint64_t(a.row0 + split) * M + uint64_t(tile) * TB);
    #pragma unroll
    for (int v = 0; v < MAC_VPT; ++v)
        __stcg(&yp[tid + v * T], acc[v]);

    /* ticket: the last CTA of this job to get here finishes the frame */
    __threadfence();
    __syncthreads();
    if (tid == 0)
    {
        uint32_t old    = atomicAdd(&tickets[jobi], 1u);
        uint32_t last   = (old == a.splits * gridDim.y - 1) ? 1u : 0u;
        if (last)
            tickets[jobi]   = 0;                /* ready for the next launch */
        *flag           = last;
    }
    __syncthreads();
    FRAME_STAMP(2);
    if (*flag == 0)
        return;
    __threadfence();
    /* end of a pipelined tail: release the slot, then let the launch complete in stream order */
    auto tail_done = [&]()
    {
        if (!pipelined)
            return;
        __threadfence();
        __syncthreads();
        if (tid == 0)
        {
            asm volatile("st.release.gpu.global.u32 [%0], %1;" :: "l"(my_done), "r"(a.seq + 1u) : "memory");
            asm volatile("griddepcontrol.wait;" ::: "memory");
        }
    };

    /* The inverse transform is the exposed tail of the launch: twiddles go to shared memory
     * (the stage buffers are idle now) so that its dependent loads stay on chip. */
    constexpr bool TAIL_PP = (RANK <= 12);      /* two work buffers fit the (>= 2) stage buffers */
    constexpr int  TAIL_RG = (RANK <= 9) ? 8 : 4;   /* partial rows in flight per round: the small CTAs of the small
                                                       ranks have the registers, and their row sum is pure latency */
    constexpr uint32_t TAIL_WORK = C::WORK * (TAIL_PP ? 2 : 1);
    float2 *wa      = stages, *wb = TAIL_PP ? stages + C::WORK : nullptr;
    const float2 *tw = a.tw;
    if (tw_early)
        tw              = reinterpret_cast<const float2 *>(po + 3 * AW);     /* there since the forward transform */
    else if (TAIL_WORK + uint32_t(C::TW_TOTAL) <= NS * 2 * stage_elems)
    {
        float2 *tws     = stages + TAIL_WORK;
        for (uint32_t i = tid; i < uint32_t(C::TW_TOTAL); i += T)
            tws[i]          = a.tw[i];
        tw              = tws;                  /* visible after inv_body's first barrier */
    }
    if (GEN || (ra.mode == 0))
    {
        if (GEN && spread)
        {
            /* the spread answers (see above): every CTA of the job is past its ticket.  They and
             * the samples of P2 travel to shared memory UNDER the inverse transform. */
            for (uint32_t i = tid; i < job.n; i += T)
                cp_async4(po + i, ans1 + i);
            for (uint32_t i = tid; i < job.n2; i += T)
            {
                cp_async4(po + AW + i, ans2 + i);
                cp_async4(po + 2 * AW + i, job.psrc2 + i);
            }
        }
        /* lookahead: the block's tail T, split rows written by the K launches before this one */
        const float2 *yT    = nullptr;
        uint32_t nT         = 0;
        if ((LK != 0) && a.la_use)
        {
            if (tid == 0)
                wait_ge<false>(a.la_prod + size_t(a.la_get) * a.n_cap + job.inst, a.la_get_need, a.error, SPIN_ERR_RING);
            __syncthreads();
            yT                  = a.la_T + ((uint64_t(a.la_get) * a.n_jobs + jobi) * LK + a.la_c) * a.splits * M;
            nT                  = a.splits;
            FRAME_STAMP(7);
        }
        inv_body<RANK, TAIL_PP, TAIL_RG, int(T)>(wa, wb, ysum, nsum, job.dst, a.tw, tw, false, int(tid),
                                                 -1, nullptr, nullptr, yT, nT);
        if (nT != 0)
        {
            /* the T rows have been read: the buffer may take the next group's tails */
            __threadfence();
            __syncthreads();
            if (tid == 0)
                asm volatile("red.release.gpu.global.add.u32 [%0], 1;"
                             :: "l"(a.la_cons + size_t(a.la_get) * a.n_cap + job.inst) : "memory");
        }
        if (GEN)
            FRAME_STAMP(7);
        if (GEN && spread)
        {
            cp_async_wait_all();
            __syncthreads();
            for (uint32_t i = tid; i < job.n; i += T)
                job.pdst[i]         = po[i];
            for (uint32_t i = tid; i < job.n2; i += T)
            {
                d.cur[job.off2 + i] = po[2 * AW + i];
                job.pdst2[i]        = job.dst[job.off2 + i] + po[AW + i];
            }
        }
        else if (GEN && (job.n2 > 0))
        {
            /* P2: the first samples of the frame that has just started, answered from the block
             * (job.dst = the instance's pending block) the inverse transform has just produced */
            __syncthreads();
            for (uint32_t i = tid; i < job.n2; i += T)
                d.cur[job.off2 + i] = job.psrc2[i];
            __syncthreads();
            partial_outputs(d.cur, d.head, job.dst, job.pdst2, job.off2, 0, job.n2, tid, T, po);
        }
        FRAME_STAMP(3);
        tail_done();
        return;
    }

    /* ---- partition-range shard: all-to-all sum of the partial blocks over NVLink ---- */
    const uint32_t F        = ra.frame;
    const uint32_t W        = ra.world, g = ra.grank;
    const uint32_t ch       = job.inst;
    const uint32_t blk      = job.tlo - ra.t0;          /* block number since the ranks connected */
    const uint32_t s        = blk % uint32_t(REDUCE_DEPTH);
    const uint32_t seq      = blk + 1u;
    const size_t   word_of_g = ((size_t(s) * W + g) * ra.channels + ch) * F;   /* same offset in every rank's buffer */

    /* slot s is free on rank p once p has consumed block blk - DEPTH of this channel */
    if ((tid < W) && (tid != g) && (blk >= uint32_t(REDUCE_DEPTH)))
        wait_ge<true>(ra.consumed[g] + size_t(tid) * ra.channels + ch, blk - uint32_t(REDUCE_DEPTH) + 1u,
                      a.error, SPIN_ERR_PEER);
    __syncthreads();

    float *mine             = ra.scratch + size_t(ch) * F;
    FRAME_STAMP(4);
    inv_body<RANK, TAIL_PP, TAIL_RG, int(T)>(wa, wb, ysum, nsum, mine, a.tw, tw, false, int(tid));
    __syncthreads();
    FRAME_STAMP(5);

    /* send: two samples and their sequence numbers per 16-byte store, to every peer */
    for (uint32_t i = tid; i < F / 2; i += T)
    {
        const float2 v      = reinterpret_cast<const float2 *>(mine)[i];
        const uint32_t b0   = __float_as_uint(v.x), b1 = __float_as_uint(v.y);
        for (uint32_t p = 0; p < W; ++p)
            if (p != g)
                asm volatile("st.volatile.global.v4.u32 [%0], {%1, %2, %3, %4};"
                             :: "l"(ra.words[p] + word_of_g + 2 * i), "r"(b0), "r"(seq), "r"(b1), "r"(seq) : "memory");
    }

    FRAME_STAMP(6);
    /* receive and add in rank order (bit-identical on every rank) */
    {
        const uint64_t deadline = global_ns() + SPIN_LIMIT_NS;
        const bool dst8     = (reinterpret_cast<uintptr_t>(job.dst) & 7) == 0;
        for (uint32_t i = tid; i < F / 2; i += T)
        {
            float2 sum          = make_float2(0.0f, 0.0f);
            for (uint32_t p = 0; p < W; ++p)
            {
                float2 v;
                if (p == g)
                    v                   = reinterpret_cast<const float2 *>(mine)[i];
                else
                {
                    const uint2 *wp     = ra.words[g] + ((size_t(s) * W + p) * ra.channels + ch) * F + 2 * i;
                    uint32_t b0, s0, b1, s1;
                    for (uint32_t spins = 1; ; ++spins)
                    {
                        asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];"
                                     : "=r"(b0), "=r"(s0), "=r"(b1), "=r"(s1) : "l"(wp) : "memory");
                        if ((s0 == seq) && (s1 == seq))
                            break;
                        if (((spins & 255u) == 0) && (global_ns() > deadline))
                        {
                            spin_fail(a.error, SPIN_ERR_PEER);
                            break;
                        }
                    }
                    v                   = make_float2(__uint_as_float(b0), __uint_as_float(b1));
                }
                sum.x              += v.x;
                sum.y              += v.y;
            }
            if (dst8)
                reinterpret_cast<float2 *>(job.dst)[i] = sum;
            else
            {
                job.dst[2 * i]      = sum.x;
                job.dst[2 * i + 1]  = sum.y;
            }
        }
    }
    __syncthreads();
    if ((tid < W) && (tid != g))
        asm volatile("st.relaxed.sys.global.u32 [%0], %1;"
                     :: "l"(ra.consumed[tid] + size_t(g) * ra.channels + ch), "r"(seq) : "memory");
    FRAME_STAMP(3);
    tail_done();
}

template <int RANK>
__global__ void __launch_bounds__(FrameCfg<RANK>::T, FrameCfg<RANK>::MINB)
k_frame(const StepArgs a, const MacShape sh, uint32_t *tickets, const ReduceArgs ra)
{
    frame_body<RANK, false>(a, sh, tickets, ra, nullptr);
}

/* the job-list form; a.jobs == NULL: the (at most JOB_PACK) jobs are in `pack` */
template <int RANK>
__global__ void __launch_bounds__(FrameCfg<RANK>::T, FrameCfg<RANK>::MINB)
k_frame_gen(const StepArgs a, const MacShape sh, uint32_t *tickets, const __grid_constant__ JobPack pack)
{
    ReduceArgs ra;
    ra.mode = 0;
    frame_body<RANK, true>(a, sh, tickets, ra, pack.j);
}

/* ------------------------------------------------------------------------------------------- */
/* Partial-call path (calls that do not complete whole frames, or a non-zero phase)              */

/* cur[off .. off+n) = psrc[0 .. n)   (first half of a large P1 segment; k_partial follows) */
__global__ void k_store(const StepArgs a)
{
    for (uint32_t jb = blockIdx.y; jb < a.n_jobs; jb += gridDim.y)
    {
        const Job job       = a.jobs[jb];
        float *cur          = a.inst[job.inst].cur;
        for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < job.n; i += gridDim.x * blockDim.x)
            cur[job.off + i]    = job.psrc[i];
    }
}

/* pdst[i] = pend[off + i] + own-frame term, i < n: grid.x CTAs share the outputs of one job
 * (after k_store: only `cur` is read, so pdst == psrc is safe). */
__global__ void __launch_bounds__(256)
k_partial(const StepArgs a)
{
    __shared__ float po[PO_SMEM_FLOATS];
    for (uint32_t jb = blockIdx.y; jb < a.n_jobs; jb += gridDim.y)
    {
        const Job job       = a.jobs[jb];
        const InstDesc &d   = a.inst[job.inst];
        const uint32_t per  = (job.n + gridDim.x - 1) / gridDim.x;
        const uint32_t i0   = min(job.n, blockIdx.x * per), i1 = min(job.n, i0 + per);
        partial_outputs(d.cur, d.head, d.pend, job.pdst, job.off, i0, i1, threadIdx.x, blockDim.x, po);
    }
}

/* Both in ONE launch for steps in which no frame completes (a call inside a frame): one CTA per
 * job stores the samples and answers them. */
__global__ void __launch_bounds__(256)
k_partial_fused(const StepArgs a, const __grid_constant__ JobPack pack)
{
    __shared__ float po[PO_SMEM_FLOATS];
    for (uint32_t jb = blockIdx.x; jb < a.n_jobs; jb += gridDim.x)
    {
        const Job job       = (a.jobs == nullptr) ? pack.j[jb] : a.jobs[jb];
        const InstDesc &d   = a.inst[job.inst];
        for (uint32_t i = threadIdx.x; i < job.n; i += blockDim.x)
            d.cur[job.off + i]  = job.psrc[i];
        __syncthreads();
        partial_outputs(d.cur, d.head, d.pend, job.pdst, job.off, 0, job.n, threadIdx.x, blockDim.x, po);
        __syncthreads();
    }
}

/* k_partial_tiles : the same answer for a call deep inside a LONG frame (ranks 14..16: up to 32768
 * taps per output sample), with the tap tiles spread over grid.x CTAs instead of walked one after
 * the other: CTA (t, job) sums tile t for every output of the job (fp64 partial per output, into
 * `partials` [job][tile][PT_MAXN]), the last CTA of a job to finish (ticket) adds the tiles in
 * order -- deterministic -- and delivers.  n <= PT_MAXN outputs per job; the new samples are read
 * from the caller's segment (never from `cur`), and the segment's outputs are written only after
 * every CTA has taken its ticket, so pdst == psrc is safe. */
constexpr uint32_t PT_MAXN = 256;

__global__ void __launch_bounds__(256)
k_partial_tiles(const StepArgs a, const __grid_constant__ JobPack pack, double *partials, uint32_t *tickets,
                uint32_t max_tiles)
{
    __shared__ float po[PO_SMEM_FLOATS];
    __shared__ uint32_t last;
    const uint32_t tid      = threadIdx.x, T = blockDim.x;
    const uint32_t jb       = blockIdx.y, tile = blockIdx.x;
    const Job job           = (a.jobs == nullptr) ? pack.j[jb] : a.jobs[jb];
    const InstDesc d        = a.inst[job.inst];
    const uint32_t n        = job.n, off = job.off;
    const uint32_t m_max    = off + n - 1;
    const uint32_t tiles    = m_max / PO_TILE + 1;
    if (tile >= tiles)
        return;

    uint32_t G              = 1;
    while ((G < 32) && (n * G * 2 <= T))
        G                     <<= 1;
    const uint32_t lane     = tid % G, i = tid / G;             /* one window: T / G >= n */
    const bool live         = i < n;
    float *cs               = po, *hs = po + PO_TILE;
    const uint32_t j0       = tile * PO_TILE;
    const int32_t hbase     = int32_t(off) - int32_t(j0) - int32_t(PO_TILE) + 1;
    const uint32_t hcount   = PO_TILE + n - 1;
    const uint32_t kend     = min(PO_TILE, (m_max - j0 + 4 * G) & ~(4 * G - 1));
    for (uint32_t k = tid; k < kend; k += T)
    {
        const uint32_t j        = j0 + k;
        cs[k]                   = (j < off) ? d.cur[j] : ((j <= m_max) ? job.psrc[j - off] : 0.0f);
    }
    for (uint32_t k = (PO_TILE - kend) + tid; k < hcount; k += T)
    {
        const int32_t h         = hbase + int32_t(k);
        hs[k]                   = (h >= 0) ? d.head[h] : 0.0f;
    }
    __syncthreads();
    double total            = 0.0;
    if (live)
    {
        const float *hp         = hs + i + (PO_TILE - 1);
        float p0 = 0.0f, p1 = 0.0f, p2 = 0.0f, p3 = 0.0f;
        #pragma unroll 2
        for (uint32_t k = lane; k < kend; k += 4 * G)
        {
            p0                      = fmaf(cs[k],         hp[-int32_t(k)],         p0);
            p1                      = fmaf(cs[k + G],     hp[-int32_t(k + G)],     p1);
            p2                      = fmaf(cs[k + 2 * G], hp[-int32_t(k + 2 * G)], p2);
            p3                      = fmaf(cs[k + 3 * G], hp[-int32_t(k + 3 * G)], p3);
        }
        total                   = double((p0 + p1) + (p2 + p3));
    }
    for (uint32_t sft = G >> 1; sft > 0; sft >>= 1)
        total                  += __shfl_xor_sync(0xffffffffu, total, sft);
    double *mine            = partials + (size_t(jb) * max_tiles + tile) * PT_MAXN;
    if (live && (lane == 0))
        mine[i]                 = total;

    __threadfence();
    __syncthreads();
    if (tid == 0)
    {
        const uint32_t old      = atomicAdd(&tickets[jb], 1u);
        last                    = (old == tiles - 1) ? 1u : 0u;
        if (last)
            tickets[jb]             = 0;
    }
    __syncthreads();
    if (!last)
        return;
    __threadfence();
    const double *all       = partials + size_t(jb) * max_tiles * PT_MAXN;
    for (uint32_t o = tid; o < n; o += T)
    {
        double sum              = 0.0;
        for (uint32_t t = 0; t < tiles; ++t)
            sum                    += __ldcg(all + size_t(t) * PT_MAXN + o);
        const float x           = job.psrc[o];
        job.pdst[o]             = d.pend[off + o] + float(sum);
        d.cur[off + o]          = x;
    }
}

/* ------------------------------------------------------------------------------------------- */
/* init helpers                                                                                 */

/* G[q][k] = H[q][k] + (-1)^k H[q-1][k],  q = 0 .. bins, H[-1] = H[bins] = 0.  Packed bin 0 is
 * (DC, Nyquist = bin M), both even, so it takes '+' like every even bin. */
__global__ void k_fold(float2 *G, const float2 *H, uint32_t bins, uint32_t M)
{
    /* grid.y strides over the rows: IRs with more than 65535 partitions exist (rank 8, minutes) */
    for (uint32_t q = blockIdx.y; q <= bins; q += gridDim.y)
    for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < M; k += gridDim.x * blockDim.x)
    {
        float2 cur      = (q < bins) ? H[uint64_t(q) * M + k] : make_float2(0.0f, 0.0f);
        float2 prev     = (q > 0) ? H[uint64_t(q - 1) * M + k] : make_float2(0.0f, 0.0f);
        float sgn       = (k & 1) ? -1.0f : 1.0f;
        G[uint64_t(q) * M + k] = make_float2(cur.x + sgn * prev.x, cur.y + sgn * prev.y);
    }
}

/* The same for many instances in one launch (batched IR ingest): instance i folds rows
 * H[h_row .. h_row + bins) into its G (bins + 1 rows) and keeps taps [0, F) in `head`. */
struct FoldDesc
{
    float2         *G;
    float          *head;           /* NULL: no time-domain head (partition-range shard with part_offset > 0) */
    uint64_t        h_row;          /* first row of this instance in the H / padded-IR slabs */
    uint32_t        bins;
    uint32_t        pad;
};

__global__ void k_fold_many(const FoldDesc *desc, uint32_t n, const float2 *H, const float *ir, uint32_t M)
{
    for (uint32_t i = blockIdx.z; i < n; i += gridDim.z)
    {
        const FoldDesc d    = desc[i];
        const float2 *Hi    = H + d.h_row * M;
        for (uint32_t q = blockIdx.y; q <= d.bins; q += gridDim.y)
        for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < M; k += gridDim.x * blockDim.x)
        {
            float2 cur      = (q < d.bins) ? Hi[uint64_t(q) * M + k] : make_float2(0.0f, 0.0f);
            float2 prev     = (q > 0) ? Hi[uint64_t(q - 1) * M + k] : make_float2(0.0f, 0.0f);
            float sgn       = (k & 1) ? -1.0f : 1.0f;
            d.G[uint64_t(q) * M + k] = make_float2(cur.x + sgn * prev.x, cur.y + sgn * prev.y);
            if ((q == 0) && (d.head != nullptr))
                d.head[k]       = ir[d.h_row * M + k];
        }
    }
}

/* dst[i] += add[i] (fastconv_apply accumulates, SURVEY a13) */
__global__ void k_accumulate(float *dst, const float *add, uint64_t total)
{
    for (uint64_t i = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
         i += uint64_t(gridDim.x) * blockDim.x)
        dst[i]     += add[i];
}

/* dsp::convolve, batched: dst[a + b] += src[a] * conv[b].  One thread per output sample gathers
 * its terms (no atomics, deterministic order). */
__global__ void k_convolve(float *dst, uint64_t dst_stride, const float *src, uint64_t src_stride,
                           const float *conv, uint64_t conv_stride, uint32_t length, uint32_t count)
{
    const float *x      = src + uint64_t(blockIdx.y) * src_stride;
    const float *h      = conv + uint64_t(blockIdx.y) * conv_stride;
    float *y            = dst + uint64_t(blockIdx.y) * dst_stride;
    const uint32_t n    = count + length - 1;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    {
        uint32_t a0     = (i >= length) ? i - length + 1 : 0;
        uint32_t a1     = (i < count) ? i : count - 1;
        float acc       = 0.0f;
        for (uint32_t a = a0; a <= a1; ++a)
            acc             = fmaf(x[a], h[i - a], acc);
        y[i]           += acc;
    }
}

/* packed spectrum product for the fastconv primitives: y = a * b, bin 0 component-wise */
__global__ void k_cmul(float2 *y, const float2 *a, const float2 *b, uint32_t M, uint64_t total)
{
    for (uint64_t i = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
         i += uint64_t(gridDim.x) * blockDim.x)
    {
        float2 u = a[i], v = b[i];
        y[i]    = ((i % M) == 0) ? make_float2(u.x * v.x, u.y * v.y) : cmul(u, v);
    }
}

} /* namespace b200conv */

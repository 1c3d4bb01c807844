/*
 * engine.cu -- host side of the batched convolver: instance table, frame bookkeeping, ring
 * indices, job lists, kernel launches, and the C ABI declared in include/b200conv.h.
 *
 * Frame bookkeeping follows lsp::dspu::Convolver (reference src/main/util/Convolver.cpp):
 * rank clamp :87, frame offset from phase :140, bins :93, zero output when not initialised
 * :219-223, zero latency for any call size :225-313.  What differs is the arithmetic plan:
 * uniform partitions in folded-overlap form, an input-spectrum ring instead of a shifted
 * time-domain tail (:304-311), one inverse FFT per frame instead of one per partition (:280-285).
 */
#include "b200conv.h"
#include "kernels.cuh"

#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <algorithm>
#include <new>
#include <string>
#include <thread>
#include <vector>

using namespace b200conv;

extern "C" int b200conv_reduce_disconnect(b200conv_batch_t *b);
extern "C" int b200conv_init_shared(b200conv_batch_t *b, size_t idx, size_t src_idx, float phase);

/* The C ABI must not leak C++ exceptions: the entry points that allocate host containers run
 * their body through a guarded shim (end of file). */

/* ------------------------------------------------------------------------------------------- */
/* errors                                                                                       */

static thread_local std::string g_last_error;

static int fail(int code, const char *fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_last_error = buf;
    return code;
}

#define CU(call)                                                                            \
    do {                                                                                    \
        cudaError_t e_ = (call);                                                            \
        if (e_ != cudaSuccess)                                                              \
            return fail((e_ == cudaErrorMemoryAllocation) ? B200CONV_ERR_NOMEM              \
                                                          : B200CONV_ERR_CUDA,             \
                        "%s failed: %s", #call, cudaGetErrorString(e_));                    \
    } while (0)

#define TRY(expr)   do { int rc_ = (expr); if (rc_ != B200CONV_OK) return rc_; } while (0)

/* ------------------------------------------------------------------------------------------- */
/* per-rank kernel dispatch                                                                     */

static const int MAX_DEVICES = 64;
static const uint32_t MAX_FEW_JOBS = 148;     /* up to this many frames per launch count as "few" (one per SM) */

/* function attributes are per device; the caller has made the batch's device current */
static int current_device()
{
    int dev = 0;
    cudaGetDevice(&dev);
    return ((dev >= 0) && (dev < MAX_DEVICES)) ? dev : 0;
}

/* k_fwd / k_inv loop over their jobs: never launch more CTAs than fit on the device at once */
static uint32_t resident_grid(uint32_t jobs, int threads, size_t smem)
{
    static int sms[MAX_DEVICES] = { 0 };
    int dev = current_device();
    if (sms[dev] == 0)
    {
        cudaDeviceProp prop;
        sms[dev] = (cudaGetDeviceProperties(&prop, dev) == cudaSuccess) ? prop.multiProcessorCount : 148;
    }
    size_t by_smem      = (227u * 1024u) / (smem + 1024u);
    size_t by_threads   = 2048u / size_t(threads);
    size_t per_sm       = (by_smem < by_threads) ? by_smem : by_threads;
    if (per_sm < 1)     per_sm = 1;
    if (per_sm > 16)    per_sm = 16;
    size_t cap          = per_sm * size_t(sms[dev]);
    return (jobs < cap) ? jobs : uint32_t(cap);
}

/* <<< >>> with the programmatic-serialisation attribute when `pdl` (the kernel then starts as soon
 * as every CTA of its predecessor in the stream has started, and orders itself with
 * griddepcontrol.wait) */
template <typename K, typename... Args>
static cudaError_t launch_k(K kernel, dim3 grid, dim3 block, size_t smem, cudaStream_t st, bool pdl, Args... args)
{
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim             = grid;
    cfg.blockDim            = block;
    cfg.dynamicSmemBytes    = smem;
    cfg.stream              = st;
    cudaLaunchAttribute attr[1];
    attr[0].id              = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = pdl ? 1 : 0;
    cfg.attrs               = attr;
    cfg.numAttrs            = 1;
    return cudaLaunchKernelEx(&cfg, kernel, args...);
}

static uint32_t rows_per_job_host(const StepArgs &a)
{
    return (a.rows != 0) ? a.rows : a.splits;
}

template <int RANK>
static cudaError_t launch_fwd_r(const StepArgs &a, uint32_t grid, cudaStream_t st, bool pdl)
{
    using C = FftCfg<RANK>;
    static bool attr_set[MAX_DEVICES] = { false };
    int dev = current_device();
    if ((!attr_set[dev]) && (C::SMEM > 48 * 1024))
    {
        cudaError_t e = cudaFuncSetAttribute(k_fwd<RANK>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(C::SMEM));
        if (e != cudaSuccess)
            return e;
    }
    attr_set[dev] = true;
    if constexpr (C::PP)
    {
        /* many jobs per CTA and device-resident input: prefetch the next job's input (k_fwd_staged) */
        constexpr size_t SS = StageCfg<RANK>::FWD_SMEM;
        const uint32_t cap  = resident_grid(grid, C::T, SS);
        if ((grid >= 2 * cap) && !(a.flags & STEP_HOST_IO) && (!pdl))
        {
            static bool attr_staged[MAX_DEVICES] = { false };
            if ((!attr_staged[dev]) && (SS > 48 * 1024))
            {
                cudaError_t e = cudaFuncSetAttribute(k_fwd_staged<RANK>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(SS));
                if (e != cudaSuccess)
                    return e;
            }
            attr_staged[dev] = true;
            k_fwd_staged<RANK><<<cap, C::T, SS, st>>>(a);      /* (never part of a programmatic chain) */
            return cudaGetLastError();
        }
    }
    if constexpr (!C::PP)
    {
        /* few frames at a big rank: one CTA per half frame (k_fwd_half); rank 16 always, its two
         * halves would otherwise run one after the other in the same CTA */
        using H = FftCfg<RANK, 0, 1>;
        if ((RANK >= 16) || (grid <= 2 * MAX_FEW_JOBS))
        {
            static bool attr_half[MAX_DEVICES] = { false };
            if ((!attr_half[dev]) && (H::SMEM > 48 * 1024))
            {
                cudaError_t e = cudaFuncSetAttribute(k_fwd_half<RANK>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(H::SMEM));
                if (e != cudaSuccess)
                    return e;
            }
            attr_half[dev] = true;
            return launch_k(k_fwd_half<RANK>, dim3(resident_grid(2 * grid, H::T, H::SMEM)), dim3(H::T), H::SMEM, st, pdl, a);
        }
    }
    return launch_k(k_fwd<RANK>, dim3(resident_grid(grid, C::T, C::SMEM)), dim3(C::T), C::SMEM, st, pdl, a);
}

template <int RANK, int RG>
static cudaError_t launch_inv_rg(const StepArgs &a, uint32_t grid, cudaStream_t st, bool pdl)
{
    using C = FftCfg<RANK>;
    static bool attr_set[MAX_DEVICES] = { false };
    int dev = current_device();
    if ((!attr_set[dev]) && (C::SMEM > 48 * 1024))
    {
        cudaError_t e = cudaFuncSetAttribute(k_inv<RANK, RG>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(C::SMEM));
        if (e != cudaSuccess)
            return e;
    }
    attr_set[dev] = true;
    return launch_k(k_inv<RANK, RG>, dim3(resident_grid(grid, C::T, C::SMEM)), dim3(C::T), C::SMEM, st, pdl, a);
}

template <int RANK>
static cudaError_t launch_inv_r(const StepArgs &a, uint32_t grid, cudaStream_t st, bool pdl, uint32_t *tickets)
{
    using C = FftCfg<RANK>;
    if constexpr (C::PP)
    {
        /* one partial row per job and many jobs per CTA: prefetch the next row (k_inv_staged) */
        constexpr size_t SS = StageCfg<RANK>::INV_SMEM;
        const uint32_t cap  = resident_grid(grid, C::T, SS);
        if ((rows_per_job_host(a) == 1) && (grid >= 2 * cap) && ((reinterpret_cast<uintptr_t>(a.ypart) & 15) == 0) && (!pdl))
        {
            static bool attr_staged[MAX_DEVICES] = { false };
            int dev = current_device();
            if ((!attr_staged[dev]) && (SS > 48 * 1024))
            {
                cudaError_t e = cudaFuncSetAttribute(k_inv_staged<RANK>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(SS));
                if (e != cudaSuccess)
                    return e;
            }
            attr_staged[dev] = true;
            k_inv_staged<RANK><<<cap, C::T, SS, st>>>(a);
            return cudaGetLastError();
        }
    }
    if constexpr (!C::PP)
    {
        /* few frames at a big rank: one CTA per half frame, then an element-wise combine */
        using H = FftCfg<RANK, 0, 1>;
        if ((a.park != nullptr) && ((RANK >= 16) || (grid <= 2 * MAX_FEW_JOBS)))
        {
            static bool attr_half[MAX_DEVICES] = { false };
            int dev = current_device();
            if ((!attr_half[dev]) && (H::SMEM > 48 * 1024))
            {
                cudaError_t e = cudaFuncSetAttribute(k_inv_half<RANK>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(H::SMEM));
                if (e != cudaSuccess)
                    return e;
            }
            attr_half[dev] = true;
            /* with a ticket array the second half to finish combines; otherwise an element-wise launch */
            cudaError_t e = launch_k(k_inv_half<RANK>, dim3(resident_grid(2 * grid, H::T, H::SMEM)), dim3(H::T),
                                     H::SMEM, st, pdl, a, tickets);
            if ((e != cudaSuccess) || (tickets != nullptr))
                return e;
            const uint32_t F = 1u << (RANK - 1);
            dim3 cg((F / 256 < 32) ? F / 256 : 32, (grid < 4096) ? grid : 4096);
            return launch_k(k_inv_combine, cg, dim3(256), 0, st, pdl, a);
        }
    }
    /* the row-group size only matters on the ping-pong ranks (FftCfg::PP) */
    if (FftCfg<RANK>::PP && (rows_per_job_host(a) <= 2))
        return launch_inv_rg<RANK, 2>(a, grid, st, pdl);
    return launch_inv_rg<RANK, 8>(a, grid, st, pdl);
}

#define RANK_SWITCH(fn, rank, ...)                                      \
    switch (rank) {                                                     \
        case 8:  return fn<8>(__VA_ARGS__);                             \
        case 9:  return fn<9>(__VA_ARGS__);                             \
        case 10: return fn<10>(__VA_ARGS__);                            \
        case 11: return fn<11>(__VA_ARGS__);                            \
        case 12: return fn<12>(__VA_ARGS__);                            \
        case 13: return fn<13>(__VA_ARGS__);                            \
        case 14: return fn<14>(__VA_ARGS__);                            \
        case 15: return fn<15>(__VA_ARGS__);                            \
        case 16: return fn<16>(__VA_ARGS__);                            \
        default: return cudaErrorInvalidValue;                          \
    }

/* `jobs` frame transforms (the kernels loop over them with a resident grid) */
static cudaError_t launch_fwd(const StepArgs &args, uint32_t jobs, cudaStream_t st, bool pdl = false)
{
    StepArgs a  = args;
    a.n_jobs    = jobs;
    RANK_SWITCH(launch_fwd_r, a.rank, a, jobs, st, pdl)
}

/* tickets: one zeroed counter per job (NULL: none available) -- lets the half-frame inverse of the
 * big ranks combine its halves itself */
static cudaError_t launch_inv(const StepArgs &args, uint32_t jobs, cudaStream_t st, bool pdl = false,
                              uint32_t *tickets = nullptr)
{
    StepArgs a  = args;
    a.n_jobs    = jobs;
    RANK_SWITCH(launch_inv_r, a.rank, a, jobs, st, pdl, tickets)
}

struct MacPlan
{
    MacShape    sh;
    uint32_t    tiles, threads, splits;
    size_t      smem;
};

static int g_tune_tile = 0;         /* developer option "mac_tile": bins per k_mac CTA at ranks >= 14 (0 = 1024) */

static MacPlan plan_mac(uint32_t rank, uint32_t jobs, uint32_t max_nq, int sm_count,
                        int tune_splits, int tune_stages)
{
    MacPlan p;
    uint32_t M      = 1u << (rank - 1);
    p.sh.TB         = (M < 1024) ? M : 1024;
    if ((rank >= 14) && (g_tune_tile > 0))
        p.sh.TB         = uint32_t(g_tune_tile);
    p.sh.QB         = 1024 / p.sh.TB;
    p.sh.NS         = (tune_stages > 0) ? uint32_t(tune_stages) : 2;      /* measured: 2 x 16 KiB beats 3 (profiles/) */
    p.tiles         = M / p.sh.TB;
    p.threads       = p.sh.TB / (2 * MAC_VPT);
    p.sh.bias       = 0;
    p.smem          = size_t(2) * p.sh.NS * p.sh.QB * p.sh.TB * sizeof(float2) + p.sh.NS * sizeof(uint64_t) + 16;

    uint32_t splits;
    if (tune_splits > 0)
        splits          = uint32_t(tune_splits);
    else
    {
        /* aim at ~3.5 co-resident CTAs per SM so that all chunks stream concurrently (4 fit) */
        uint32_t target = (7u * uint32_t(sm_count)) / 2u;
        uint32_t ctas   = jobs * p.tiles;
        splits          = (ctas > 0) ? (target / ctas) : 1;
    }
    uint32_t cap    = max_nq / (2 * p.sh.QB);           /* at least two stages of work per chunk */
    if (splits > cap)   splits = cap;
    if (splits > 32)    splits = 32;
    if (splits < 1)     splits = 1;
    p.splits        = splits;
    /* (deeper stage rings for small, latency-bound grids were measured and bought nothing:
     * tools/ab_stages.py, 2 / 3 / 4 stages within 1 % on cfg 1 and cfg 2, two stages 5-8 % ahead at
     * 8 channels per GPU) */
    return p;
}

static cudaError_t launch_mac_raw(const StepArgs &a, const MacPlan &p, uint32_t jobs, cudaStream_t st,
                                  bool pdl = false)
{
    static size_t attr_smem[MAX_DEVICES] = { 0 };
    int dev = current_device();
    if (p.smem > attr_smem[dev])
    {
        cudaError_t e = cudaFuncSetAttribute(k_mac, cudaFuncAttributeMaxDynamicSharedMemorySize, int(p.smem));
        if (e != cudaSuccess)
            return e;
        attr_smem[dev] = p.smem;
    }
    dim3 grid(jobs * p.splits, p.tiles);
    if (pdl)
    {
        /* may start while the preceding k_frame launch is in its tail (STEP_WAIT_HEAD) */
        cudaLaunchConfig_t cfg;
        memset(&cfg, 0, sizeof(cfg));
        cfg.gridDim             = grid;
        cfg.blockDim            = dim3(p.threads);
        cfg.dynamicSmemBytes    = p.smem;
        cfg.stream              = st;
        cudaLaunchAttribute attr[1];
        attr[0].id              = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs               = attr;
        cfg.numAttrs            = 1;
        return cudaLaunchKernelEx(&cfg, k_mac, a, p.sh);
    }
    k_mac<<<grid, p.threads, p.smem, st>>>(a, p.sh);
    return cudaGetLastError();
}

template <int TF>
static cudaError_t launch_mac_multi_t(const StepArgs &a, const MacPlan &p, uint32_t jobs, cudaStream_t st)
{
    static size_t attr_smem[MAX_DEVICES] = { 0 };
    int dev = current_device();
    if (p.smem > attr_smem[dev])
    {
        cudaError_t e = cudaFuncSetAttribute(k_mac_multi<TF>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(p.smem));
        if (e != cudaSuccess)
            return e;
        attr_smem[dev] = p.smem;
    }
    dim3 grid(jobs * p.splits, p.tiles);
    /* TB/2 consumer threads (one float4 column each) + one producer warp */
    k_mac_multi<TF><<<grid, p.sh.TB / 2 + 32, p.smem, st>>>(a, p.sh);
    return cudaGetLastError();
}

static cudaError_t launch_mac_multi(const StepArgs &a, const MacPlan &p, uint32_t jobs, uint32_t tf, cudaStream_t st)
{
    switch (tf)
    {
        case 2:  return launch_mac_multi_t<2>(a, p, jobs, st);
        case 4:  return launch_mac_multi_t<4>(a, p, jobs, st);
        case 8:  return launch_mac_multi_t<8>(a, p, jobs, st);
        default: return cudaErrorInvalidValue;
    }
}

template <int RANK>
static cudaError_t launch_frame_r(const StepArgs &a, const MacPlan &p, uint32_t jobs, uint32_t *tickets,
                                  const ReduceArgs &ra, bool pdl, cudaStream_t st)
{
    static size_t attr_smem[MAX_DEVICES] = { 0 };
    int dev = current_device();
    if (p.smem > attr_smem[dev])
    {
        cudaError_t e = cudaFuncSetAttribute(k_frame<RANK>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(p.smem));
        if (e != cudaSuccess)
            return e;
        attr_smem[dev] = p.smem;
    }
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim             = dim3(jobs * p.splits, p.tiles);
    cfg.blockDim            = dim3(p.threads);
    cfg.dynamicSmemBytes    = p.smem;
    cfg.stream              = st;
    cudaLaunchAttribute attr[1];
    attr[0].id              = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = pdl ? 1 : 0;
    cfg.attrs               = attr;
    cfg.numAttrs            = 1;
    return cudaLaunchKernelEx(&cfg, k_frame<RANK>, a, p.sh, tickets, ra);
}

/* the job-list form (general path): no cross-GPU reduce; with `pdl` its prologue (and the launch
 * latency) hides under the tail of the launch before it -- every CTA then waits for that launch */
template <int RANK>
static cudaError_t launch_frame_gen_r(const StepArgs &a, const MacPlan &p, uint32_t jobs, uint32_t *tickets,
                                      const JobPack &pack, bool pdl, cudaStream_t st)
{
    static size_t attr_smem[MAX_DEVICES] = { 0 };
    int dev = current_device();
    if (p.smem > attr_smem[dev])
    {
        cudaError_t e = cudaFuncSetAttribute(k_frame_gen<RANK>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(p.smem));
        if (e != cudaSuccess)
            return e;
        attr_smem[dev] = p.smem;
    }
    return launch_k(k_frame_gen<RANK>, dim3(jobs * p.splits, p.tiles), dim3(p.threads), p.smem, st, pdl, a, p.sh, tickets, pack);
}

static cudaError_t launch_frame_gen(const StepArgs &a, const MacPlan &p, uint32_t jobs, uint32_t *tickets,
                                    const JobPack &pack, bool pdl, cudaStream_t st)
{
    switch (a.rank)
    {
        case 8:  return launch_frame_gen_r<8>(a, p, jobs, tickets, pack, pdl, st);
        case 9:  return launch_frame_gen_r<9>(a, p, jobs, tickets, pack, pdl, st);
        case 10: return launch_frame_gen_r<10>(a, p, jobs, tickets, pack, pdl, st);
        case 11: return launch_frame_gen_r<11>(a, p, jobs, tickets, pack, pdl, st);
        case 12: return launch_frame_gen_r<12>(a, p, jobs, tickets, pack, pdl, st);
        case 13: return launch_frame_gen_r<13>(a, p, jobs, tickets, pack, pdl, st);
        default: return cudaErrorInvalidValue;
    }
}

static cudaError_t launch_frame(const StepArgs &a, const MacPlan &p, uint32_t jobs, uint32_t *tickets,
                                const ReduceArgs &ra, bool pdl, cudaStream_t st)
{
    switch (a.rank)
    {
        case 8:  return launch_frame_r<8>(a, p, jobs, tickets, ra, pdl, st);
        case 9:  return launch_frame_r<9>(a, p, jobs, tickets, ra, pdl, st);
        case 10: return launch_frame_r<10>(a, p, jobs, tickets, ra, pdl, st);
        case 11: return launch_frame_r<11>(a, p, jobs, tickets, ra, pdl, st);
        case 12: return launch_frame_r<12>(a, p, jobs, tickets, ra, pdl, st);
        case 13: return launch_frame_r<13>(a, p, jobs, tickets, ra, pdl, st);
        default: return cudaErrorInvalidValue;
    }
}

/* ------------------------------------------------------------------------------------------- */
/* twiddle tables: exp(-2 pi i j / N), j < N, computed in double                                 */

static int make_twiddles(uint32_t rank, float2 **out)
{
    /* layout: FftCfg<RANK> in kernels.cuh (radix-4 passes | w_M^m | w_N^k), all from double */
    const size_t N = size_t(1) << rank, M = N / 2, P = M / 2;
    const size_t ns0 = ((rank - 2) & 1) ? 2 : 1;
    std::vector<float2> h;
    h.reserve(3 * P + 2);
    auto root = [](double num, double den)
    {
        double ang = -2.0 * M_PI * num / den;
        return make_float2(float(cos(ang)), float(sin(ang)));
    };
    for (size_t ns = ns0; ns < P; ns <<= 2)
        for (size_t r = 1; r <= 3; ++r)
            for (size_t k = 0; k < ns; ++k)
                h.push_back(root(double(k * r), double(4 * ns)));
    for (size_t m = 0; m < P; ++m)
        h.push_back(root(double(m), double(M)));
    for (size_t k = 0; k <= M / 2; ++k)
        h.push_back(root(double(k), double(N)));

    float2 *d = nullptr;
    CU(cudaMalloc(&d, h.size() * sizeof(float2)));
    cudaError_t e = cudaMemcpy(d, h.data(), h.size() * sizeof(float2), cudaMemcpyHostToDevice);
    if (e != cudaSuccess)
    {
        cudaFree(d);
        return fail(B200CONV_ERR_CUDA, "twiddle upload failed: %s", cudaGetErrorString(e));
    }
    *out = d;
    return B200CONV_OK;
}

/* ------------------------------------------------------------------------------------------- */
/* k_frame launches in flight, per stream                                                       */
/*                                                                                             */
/* A k_frame launch carries the programmatic-serialisation attribute, so it may become resident   */
/* while earlier k_frame launches of the SAME stream -- of this batch or of another one -- are    */
/* still in their inverse-transform tails.  Reading the caller's input block that early           */
/* (STEP_EARLY_SRC: the transform does not wait for griddepcontrol.wait, which takes the          */
/* transform out of the launch-to-launch dependency chain) is safe only if no launch that may     */
/* still be running writes that block.  This table remembers the output ranges of the k_frame     */
/* launches enqueued on a stream since its last full dependency (any other operation this library  */
/* enqueues there, or a host synchronisation); a launch whose input overlaps one of them keeps the */
/* in-kernel wait.  An early transform also writes ring slot (-t) mod S, last read by the launch    */
/* RING_SPARE + 1 blocks ago: after FRAME_CHAIN_MAX (< RING_SPARE) launches in a row an            */
/* early-capable launch is launched WITHOUT the attribute (a full dependency), which bounds the     */
/* table and proves that reader complete.  Launches that keep the in-kernel wait need no bound.     */

namespace
{
    const uint32_t FRAME_CHAIN_MAX = 24;

    /* the rows of one block in a planar matrix: row i covers [lo + i * stride, + len) bytes */
    struct BlockRows
    {
        uintptr_t   lo;
        size_t      stride, len, rows;
        uintptr_t hi() const    { return lo + ((rows > 0) ? (rows - 1) * stride : 0) + len; }
    };

    bool rows_overlap(const BlockRows &a, const BlockRows &b)
    {
        if ((a.lo >= b.hi()) || (b.lo >= a.hi()))
            return false;
        if ((a.stride == b.stride) && (a.stride >= a.len) && (a.stride >= b.len) && (a.stride > 0))
        {
            /* two column blocks of matrices with one row pitch: compare the column offsets */
            const size_t d  = (b.lo >= a.lo) ? (b.lo - a.lo) % a.stride : (a.stride - (a.lo - b.lo) % a.stride) % a.stride;
            return (d < a.len) || (d + b.len > a.stride);
        }
        return true;                        /* different pitches: the enclosing intervals decide */
    }

    struct FrameHistory
    {
        cudaStream_t    st      = nullptr;
        int             dev     = -1;
        uint32_t        n       = 0;        /* > FRAME_CHAIN_MAX: more launches in flight than the table holds */
        uint64_t        stamp   = 0;
        BlockRows       out[FRAME_CHAIN_MAX], in[FRAME_CHAIN_MAX];
    };
    std::mutex      g_hist_lock;
    FrameHistory    g_hist[32];
    uint64_t        g_hist_clock = 0;

    FrameHistory *hist_find(cudaStream_t st, int dev, bool create)
    {
        FrameHistory *lru = &g_hist[0];
        for (FrameHistory &h : g_hist)
        {
            if ((h.dev == dev) && (h.st == st))
                return &h;
            if (h.stamp < lru->stamp)
                lru     = &h;
        }
        if (!create)
            return nullptr;
        /* an evicted entry is forgotten: its stream's next launch finds no history, which is safe
         * only because eviction makes that launch conservative (n = FRAME_CHAIN_MAX + 1) */
        lru->st     = st;
        lru->dev    = dev;
        lru->n      = FRAME_CHAIN_MAX + 1;
        return lru;
    }

    /* a full dependency has been (or is about to be) enqueued on `st`, or `st` was synchronised */
    void hist_reset(cudaStream_t st, int dev)
    {
        std::lock_guard<std::mutex> lock(g_hist_lock);
        FrameHistory *h = hist_find(st, dev, false);
        if (h != nullptr)
            h->n        = 0;
    }

    /* Kernels that let their successor start early (griddepcontrol.launch_dependents) but are not
     * registered below -- the job-list form, the three-kernel blocks of ranks 14..16, multi-frame
     * passes -- have been enqueued on `st`: what they write is unknown to the table, so the next
     * k_frame launch there is launched without the attribute (it starts when they have completed). */
    void hist_unknown(cudaStream_t st, int dev)
    {
        std::lock_guard<std::mutex> lock(g_hist_lock);
        FrameHistory *h = hist_find(st, dev, true);
        h->stamp        = ++g_hist_clock;
        h->n            = FRAME_CHAIN_MAX + 1;
    }

    /* Registers a k_frame launch that reads the block `in` and writes the block `out`.  `capable`:
     * the launch would like to transform its input early.  *early: it may (no launch in flight
     * writes its input); *serial: launch it without programmatic serialisation (asked of a capable
     * launch every FRAME_CHAIN_MAX, and of any launch when the table does not know what is in
     * flight: hist_unknown, an evicted entry); *dst_clash: a launch that may be in flight writes OR READS (part of) `out`
     * -- this launch must not write before those have completed. */
    void hist_launch(cudaStream_t st, int dev, bool capable, const BlockRows &in, const BlockRows &out,
                     bool *early, bool *serial, bool *dst_clash)
    {
        std::lock_guard<std::mutex> lock(g_hist_lock);
        FrameHistory *h = hist_find(st, dev, true);
        h->stamp        = ++g_hist_clock;
        *serial         = (capable && (h->n >= FRAME_CHAIN_MAX)) || (h->n > FRAME_CHAIN_MAX);
        if (*serial)
            h->n            = 0;
        bool clash      = (h->n > FRAME_CHAIN_MAX), wclash = clash;
        for (uint32_t i = 0; (i < h->n) && (i < FRAME_CHAIN_MAX); ++i)
        {
            clash          |= rows_overlap(h->out[i], in);
            wclash         |= rows_overlap(h->out[i], out) || rows_overlap(h->in[i], out);
        }
        *early          = capable && (!clash);
        *dst_clash      = wclash;
        if (h->n < FRAME_CHAIN_MAX)
        {
            h->out[h->n]    = out;
            h->in[h->n]     = in;
        }
        if (h->n <= FRAME_CHAIN_MAX)
            h->n           += 1;
    }
}

/* ------------------------------------------------------------------------------------------- */
/* batch                                                                                        */

struct Slab                         /* one device allocation shared by the instances of one init call */
{
    void       *base        = nullptr;
    size_t      refs        = 0;
};
static void slab_release(Slab *s);

struct Instance
{
    bool        active      = false;
    size_t      conv_size   = 0;
    size_t      rank        = 0;
    size_t      F           = 0;
    size_t      bins        = 0;
    size_t      nq          = 0;
    size_t      q_lo        = 0;
    size_t      S           = 0;
    size_t      off         = 0;        /* nFrameOff */
    size_t      off0        = 0;        /* nFrameOff right after init (from phase) */
    uint64_t    frames      = 0;
    bool        pend_valid  = false;
    float2     *G           = nullptr;
    float2     *ring        = nullptr;
    float      *aux         = nullptr;  /* cur | pend | head, F floats each */
    Slab       *slab        = nullptr;  /* != NULL: G (unless borrowed), ring and aux live in this slab */
    long        g_owner     = -1;       /* >= 0: G belongs to that instance (b200conv_init_shared) */
    size_t      g_sharers   = 0;        /* instances borrowing this one's G */
};

static const size_t JOB_RING_MAX = size_t(1) << 15;    /* job upload ring: 64 entries per instance, within these bounds */
static const size_t JOB_RING_MIN = size_t(1) << 10;
static const size_t RING_SPARE = 32;                    /* spare ring slots: frames transformed ahead of a multi-frame
                                                           MAC pass (8), and k_frame launches in flight (FRAME_CHAIN_MAX) */
static_assert(FRAME_CHAIN_MAX < RING_SPARE, "k_frame launches in flight must fit the spare ring slots");
static const uint64_t EARLY_MAX_BYTES = 450000000ull;  /* launches that stream more than this per block (~70 us) keep the
                                                           in-kernel wait: they hide the chain anyway, and spare themselves
                                                           the serialised launch every FRAME_CHAIN_MAX blocks */
static const uint64_t LA_MIN_BYTES = 64000000ull;      /* k_frame lookahead: only launches that stream at least this per
                                                           block (bandwidth-bound); shorter ones are latency-bound and
                                                           would only pay for the extra T rows in their tail */
static const size_t PART_MAX   = 1024;                  /* samples one P1 / P2 segment of a fused step answers */

struct b200conv_batch
{
    int                     device      = 0;
    int                     sm_count    = 148;
    size_t                  n           = 0;
    std::vector<Instance>   inst;
    size_t                  rank        = 0;        /* shared clamped rank, 0 = none active */
    cudaStream_t            stream      = nullptr;
    cudaEvent_t             ev_last     = nullptr;  /* end of the latest process_device call on a CALLER's stream */
    bool                    last_foreign = false;   /* ... and whether there was one since the last quiesce      */

    std::vector<InstDesc>   h_desc;
    InstDesc               *d_desc      = nullptr;
    std::vector<uint32_t>   active;
    uint32_t               *d_active    = nullptr;
    bool                    desc_dirty  = true;
    uint64_t                t_batch     = 0;
    size_t                  max_nq      = 0;

    float2                 *tw[B200CONV_RANK_MAX + 1] = { nullptr };
    float2                 *ypart       = nullptr;
    size_t                  ypart_bytes = 0;

    Job                    *h_jobs      = nullptr;  /* page-locked */
    Job                    *d_jobs      = nullptr;
    size_t                  job_cap     = 0;
    size_t                  job_pos     = 0;
    /* general-path scratch, sized once at create: process() never allocates (SURVEY 3.2) */
    std::vector<size_t>     g_pos;
    std::vector<Job>        g_jobs, g_fft, g_mac, g_part;
    /* IR ingest (b200conv_init_many): scratch that stays with the batch between calls */
    void                   *init_scratch = nullptr; /* device: padded taps | spectra | fold table of one round */
    size_t                  init_scratch_bytes = 0;
    float                  *init_stage[2] = { nullptr, nullptr };   /* page-locked upload staging */
    size_t                  init_stage_floats = 0;
    cudaEvent_t             init_ev[2]  = { nullptr, nullptr };
    double                 *d_partials  = nullptr;  /* k_partial_tiles: [job][tile][PT_MAXN] */
    size_t                  partials_jobs = 0;
    bool                    uniform_stale = false;  /* instances advanced one by one: t_delta must be refreshed */

    float                  *h_in = nullptr, *h_out = nullptr;   /* pinned staging */
    float                  *h_in_dev = nullptr, *h_out_dev = nullptr;  /* ... as the device addresses them */
    float                  *d_in = nullptr, *d_out = nullptr;
    size_t                  stage_floats = 0;

    b200conv_stats_t        stats       = {};
    int                     tune_splits = 0, tune_stages = 0;
    float                  *park        = nullptr;  /* k_inv_half scratch */
    size_t                  park_bytes  = 0;
    bool                    last_was_frame = false; /* the last launch on the stream was a k_frame of this batch */
    bool                    host_io     = false;    /* the running call reads / writes page-locked host matrices */
    int                     opt_fused   = 1, opt_bias = 6, opt_pdl = 1, opt_zero_copy = 1, opt_multi = 8;
    int                     opt_early_src = 1;      /* 0 never, 1 on the batch's own stream, 2 on any stream */
    uint32_t               *d_tickets   = nullptr;  /* k_frame: [FRAME_SLOTS][instances] arrival counters */
    uint32_t               *d_slot_done = nullptr;  /* k_frame: [FRAME_SLOTS][instances], see FRAME_SLOTS in kernels.cuh */
    uint32_t                frame_seq   = 0;        /* sequence number of the next k_frame launch */
    size_t                  ypart_slot_bytes = 0;   /* ypart holds FRAME_SLOTS slots of this size */
    std::vector<uint32_t>   h_slot_done;
    uint32_t               *d_ring_head = nullptr;  /* k_frame: frames published per instance; [n] = chain head (StepArgs::chain_head) */
    bool                    chain_valid = false;    /* the device word will hold chain_next once everything enqueued has run */
    uint32_t                chain_next  = 0;
    int                     opt_chain_ahead = 1;    /* ranks 14..16: the MAC of the NEXT block is launched behind this block's inverse transform */
    bool                    ahead_valid = false;    /* partitions q >= 1 of block ahead_t are (being) summed into its row slot */
    uint64_t                ahead_t     = 0;
    uint32_t                ahead_splits = 0;
    uint32_t               *h_error     = nullptr;  /* page-locked, device-mapped: a bounded in-kernel wait gave up */
    /* k_frame lookahead for one-frame calls (kernels.cuh, LA_BUFS) */
    int                     opt_lookahead = -1;     /* -1 automatic, 0 off, 2 / 4 / 8 = that group size K */
    float2                 *la_T        = nullptr;  /* [LA_BUFS][jobs][K][splits][M] */
    size_t                  la_T_bytes  = 0;
    uint32_t               *d_la_cnt    = nullptr;  /* [2][LA_BUFS][instances]: producer CTAs, consumer tails */
    bool                    la_live     = false;    /* the last launch of this batch was a lookahead k_frame (la_* below) */
    uint32_t                la_K        = 0, la_splits = 0, la_nact = 0;
    uint64_t                la_origin   = 0;        /* batch frame of the first block of the schedule (priming group) */
    uint64_t                la_next_t   = 0;        /* batch frame the next launch must carry to continue it */
    uint32_t                la_prod_cnt[LA_BUFS] = { 0 }, la_cons_cnt[LA_BUFS] = { 0 };    /* the device counters once
                                                       everything enqueued has run (same for every active instance) */
    std::vector<uint32_t>   h_ring_head;

    /* eager pending MAC for synchronous host callers: right after block t has been delivered the
     * partitions q >= 1 of block t+1 (complete frames only) are summed while the host is away,
     * so the next call only transforms its input, adds partition 0 and inverts */
    int                     opt_eager   = 1;
    int                     opt_early_pend = 1;     /* the pending MAC may start under the tail of the launch before it: 0 never, 1 auto, 2 always */
    bool                    caller_busy = false;    /* the previous pending MAC was still running when the current call arrived */
    bool                    eager_call  = false;    /* set by the synchronous entry points */
    bool                    pend_ready  = false;
    uint64_t                pend_t      = 0;        /* batch frame counter the pending rows belong to */
    uint32_t                pend_splits = 0;
    uint32_t                pend_seq    = 0;        /* sequence number of the k_frame launch the pending rows are for */
    cudaEvent_t             ev_done     = nullptr;  /* output of the current block is complete */
    cudaEvent_t             ev_pend     = nullptr;  /* the pending MAC launched after it is complete */
    bool                    pend_inflight = false;

    /* fused cross-GPU reduce (partition-range sharding) */
    ReduceArgs              reduce      = {};
    unsigned char          *xchg        = nullptr;              /* local exchange buffer (IPC shared) */
    void                   *xchg_peer[REDUCE_MAX_WORLD] = { nullptr };  /* peers' buffers, opened */
    size_t                  xchg_slots_bytes = 0, xchg_flags_off = 0, xchg_consumed_off = 0;

    bool                    profiling   = false;
    std::vector<cudaEvent_t> prof_events;           /* pairs: before / after each k_mac */
    size_t                  prof_used   = 0;
};

typedef b200conv_batch Batch;

static cudaError_t launch_mac(Batch *b, const StepArgs &a, const MacPlan &p, uint32_t jobs, cudaStream_t st,
                              bool fused = false, bool serial = false, bool chain = false)
{
    auto go = [&]() -> cudaError_t
    {
        if (fused)
        {
            const uint32_t slot = a.seq % uint32_t(FRAME_SLOTS);
            ReduceArgs ra   = b->reduce;
            if (ra.mode != 0)
                ra.scratch     += size_t(slot) * ra.channels * ra.frame;
            return launch_frame(a, p, jobs, b->d_tickets + size_t(slot) * b->n, ra,
                                (b->opt_pdl != 0) && (!b->profiling) && (!serial), st);
        }
        return launch_mac_raw(a, p, jobs, st, chain);
    };
    if (!b->profiling)
        return go();
    while (b->prof_events.size() < b->prof_used + 2)
    {
        cudaEvent_t ev;
        cudaError_t e = cudaEventCreate(&ev);
        if (e != cudaSuccess)
            return e;
        b->prof_events.push_back(ev);
    }
    cudaError_t e = cudaEventRecord(b->prof_events[b->prof_used], st);
    if (e == cudaSuccess) e = go();
    if (e == cudaSuccess) e = cudaEventRecord(b->prof_events[b->prof_used + 1], st);
    b->prof_used += 2;
    return e;
}

/* Makes the batch's device current for the duration of an API call and restores the caller's
 * device afterwards (the library must not leave a different current device behind). */
class DeviceScope
{
    private:
        int         nPrev;
        cudaError_t nErr;

    public:
        explicit DeviceScope(int device): nPrev(-1), nErr(cudaSuccess)
        {
            nErr = cudaGetDevice(&nPrev);
            if ((nErr == cudaSuccess) && (nPrev != device))
                nErr = cudaSetDevice(device);
            else
                nPrev = -1;                 /* nothing to restore */
        }
        ~DeviceScope()
        {
            if (nPrev >= 0)
                cudaSetDevice(nPrev);
        }
        cudaError_t error() const           { return nErr; }
};

#define ENTER_DEVICE(b)                                                                     \
    DeviceScope device_scope_((b)->device);                                                 \
    if (device_scope_.error() != cudaSuccess)                                               \
        return fail(B200CONV_ERR_CUDA, "cannot select device %d: %s", (b)->device,          \
                    cudaGetErrorString(device_scope_.error()))

/* Waits for everything this batch has enqueued: on its own stream and on a caller's stream.  The
 * caller's stream handle is never kept past the call that received it (the caller may destroy it);
 * an event recorded on it at the end of that call stands in for it. */
static cudaError_t quiesce(Batch *b)
{
    cudaError_t e = cudaSuccess;
    if (b->stream)
    {
        e = cudaStreamSynchronize(b->stream);
        hist_reset(b->stream, b->device);
    }
    if ((e == cudaSuccess) && b->last_foreign && (b->ev_last != nullptr))
        e = cudaEventSynchronize(b->ev_last);
    b->last_foreign = false;
    b->pend_inflight = false;
    return e;
}

/* A bounded in-kernel wait gave up (kernels.cuh, wait_ge): the results since then are garbage. */
static int check_device_error(Batch *b)
{
    const uint32_t code = (b->h_error != nullptr) ? *reinterpret_cast<volatile uint32_t *>(b->h_error) : 0u;
    if (code == 0)
        return B200CONV_OK;
    return fail(B200CONV_ERR_STATE, "an in-kernel wait timed out (%s); results since then are invalid -- "
                "re-create the batch%s", (code == SPIN_ERR_PEER) ? "a peer GPU of the fused reduce did not answer"
                                                                 : "a predecessor launch did not publish its spectrum",
                (code == SPIN_ERR_PEER) ? " and reconnect the reduce" : "");
}

static void free_instance_buffers(Instance &in)
{
    if (in.slab != nullptr)
        slab_release(in.slab);          /* the last instance of the slab frees it */
    else
    {
        if (in.G && (in.g_owner < 0))   cudaFree(in.G);
        if (in.ring)    cudaFree(in.ring);
        if (in.aux)     cudaFree(in.aux);
    }
    in.G = nullptr; in.ring = nullptr; in.aux = nullptr; in.slab = nullptr;
}

static void rebuild_tables(Batch *b)
{
    b->active.clear();
    b->max_nq   = 0;
    b->rank     = 0;
    for (size_t i = 0; i < b->n; ++i)
    {
        const Instance &in = b->inst[i];
        InstDesc &d = b->h_desc[i];
        memset(&d, 0, sizeof(d));
        if (!in.active)
            continue;
        b->active.push_back(uint32_t(i));
        b->rank     = in.rank;
        if (in.nq > b->max_nq)
            b->max_nq   = in.nq;
        d.G         = in.G;
        d.ring      = in.ring;
        d.cur       = in.aux;
        d.pend      = in.aux + in.F;
        d.head      = in.aux + 2 * in.F;
        d.t_delta   = int64_t(in.frames) - int64_t(b->t_batch);
        d.nq        = uint32_t(in.nq);
        d.q_lo      = uint32_t(in.q_lo);
        d.S         = uint32_t(in.S);
    }
    b->desc_dirty = true;
    b->pend_ready = false;
}

static int upload_tables(Batch *b, cudaStream_t st)
{
    if (!b->desc_dirty)
        return B200CONV_OK;
    hist_reset(st, b->device);          /* the copies below are full dependencies */
    b->chain_valid = false;
    b->ahead_valid = false;
    for (size_t i = 0; i < b->n; ++i)
    {
        b->h_ring_head[i]   = uint32_t(b->inst[i].frames);
        if (b->inst[i].active)
            b->h_desc[i].t_delta = int64_t(b->inst[i].frames) - int64_t(b->t_batch);
    }
    CU(cudaMemcpyAsync(b->d_ring_head, b->h_ring_head.data(), b->n * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    /* every earlier k_frame launch has completed when these copies run: all slots are free */
    for (uint32_t &v : b->h_slot_done)
        v                   = b->frame_seq;
    CU(cudaMemcpyAsync(b->d_slot_done, b->h_slot_done.data(), b->h_slot_done.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    /* ... and no lookahead tail is pending: the schedule restarts with a priming group */
    CU(cudaMemsetAsync(b->d_la_cnt, 0, 2 * LA_BUFS * b->n * sizeof(uint32_t), st));
    for (int i = 0; i < LA_BUFS; ++i)
        b->la_prod_cnt[i] = b->la_cons_cnt[i] = 0;
    b->la_live          = false;
    /* pageable sources: cudaMemcpyAsync stages them before returning */
    CU(cudaMemcpyAsync(b->d_desc, b->h_desc.data(), b->n * sizeof(InstDesc), cudaMemcpyHostToDevice, st));
    if (!b->active.empty())
        CU(cudaMemcpyAsync(b->d_active, b->active.data(), b->active.size() * sizeof(uint32_t),
                           cudaMemcpyHostToDevice, st));
    b->desc_dirty = false;
    return B200CONV_OK;
}

/* `bytes` of partial rows per launch; the buffer holds FRAME_SLOTS such slots (pipelined k_frame
 * launches rotate through them, every other user takes slot 0) */
static int ensure_ypart(Batch *b, size_t bytes, cudaStream_t st)
{
    if (bytes <= b->ypart_slot_bytes)
        return B200CONV_OK;
    CU(quiesce(b));
    CU(cudaStreamSynchronize(st));
    if (b->ypart)
        cudaFree(b->ypart);
    b->ypart        = nullptr;
    b->ypart_bytes  = 0;
    b->ypart_slot_bytes = 0;
    size_t want     = (bytes + bytes / 4 + 255) & ~size_t(255);
    CU(cudaMalloc(&b->ypart, want * FRAME_SLOTS));
    b->ypart_bytes  = want * FRAME_SLOTS;
    b->ypart_slot_bytes = want;
    b->pend_ready   = false;
    return B200CONV_OK;
}

/* the lookahead tail buffer: grown when a schedule (re)starts, never inside one */
static int ensure_la(Batch *b, size_t bytes, cudaStream_t st)
{
    if (bytes <= b->la_T_bytes)
        return B200CONV_OK;
    CU(quiesce(b));
    CU(cudaStreamSynchronize(st));
    if (b->la_T)
        cudaFree(b->la_T);
    b->la_T         = nullptr;
    b->la_T_bytes   = 0;
    b->la_live      = false;
    CU(cudaMalloc(&b->la_T, bytes));
    b->la_T_bytes   = bytes;
    return B200CONV_OK;
}

/* Group size of the k_frame lookahead for a stream of one-frame calls, from what the batch holds:
 * only launches that stream enough bytes to be bandwidth-bound, bin slices of at least 128 bins
 * (1 KiB bulk copies), and tails of at least 6K partitions (the head of 2K rows is read every block). */
static uint32_t lookahead_k(const Batch *b, uint64_t per_frame_bytes)
{
    const uint32_t M = 1u << (b->rank - 1);
    if (b->opt_lookahead >= 0)
        return uint32_t(b->opt_lookahead);
    if (per_frame_bytes < LA_MIN_BYTES)
        return 0;
    for (uint32_t k = 8; k >= 2; k >>= 1)
        if ((M / k >= 128) && (b->max_nq >= 8 * size_t(k)))
            return k;
    return 0;
}

/* What a lookahead launch copies per instance: head rows; per k_frame CTA (split x bin tile) the G
 * slices of its tail partitions and its ring window, which holds nj - 1 slices more (nj = segments
 * of the tile, kernels.cuh frame_body); the split rows of T written and read; and the 24 F bytes of
 * the transform / output of the algorithmic figure (algo_bytes). */
static uint64_t la_stream_bytes(const Instance &in, uint32_t K, bool use, const MacShape &sh, uint32_t splits)
{
    const uint64_t F  = in.F;
    const size_t q_hi = in.q_lo + in.nq;
    const size_t qs   = std::max(in.q_lo, std::min(q_hi, size_t(2) * K));
    const uint64_t nh = use ? (qs - in.q_lo) : in.nq;
    const uint32_t nt = uint32_t(q_hi - qs);
    const uint64_t W  = F / K;
    const uint64_t Wg = std::min<uint64_t>(W, sh.TB);
    const uint64_t nj = std::max<uint64_t>(1, sh.TB / W);
    uint64_t slices   = 0;
    for (uint32_t s = 0; s < splits; ++s)
    {
        uint32_t e0, e1;
        chunk_range(nt, s, splits, sh.bias, e0, e1);
        if (e1 > e0)
            slices         += 2 * uint64_t(e1 - e0) + nj - 1;
    }
    const uint64_t tail = (F / sh.TB) * slices * 8 * Wg;
    return 16 * F * nh + tail + 8 * F * splits * (use ? 2 : 1) + 8 * F;
}

static float2 *ypart_slot(const Batch *b, uint32_t seq)
{
    return reinterpret_cast<float2 *>(reinterpret_cast<unsigned char *>(b->ypart) +
                                      size_t(seq % uint32_t(FRAME_SLOTS)) * b->ypart_slot_bytes);
}

/* Ranks 13..16 with few frames per launch: scratch for the half-frame inverse transform
 * (k_inv_half, [job][2][F] floats).  Leaves a.park NULL when the launch does not qualify. */
static int attach_park(Batch *b, StepArgs &a, size_t jobs, cudaStream_t st)
{
    a.park          = nullptr;
    if ((b->rank < 13) || (jobs == 0) || ((b->rank < 16) && (jobs > 2 * MAX_FEW_JOBS)))
        return B200CONV_OK;
    const size_t bytes = jobs * (size_t(2) << (b->rank - 1)) * sizeof(float);
    if (bytes > (size_t(1) << 30))
        return B200CONV_OK;
    if (bytes > b->park_bytes)
    {
        CU(cudaStreamSynchronize(st));
        if (b->park)
            cudaFree(b->park);
        b->park         = nullptr;
        b->park_bytes   = 0;
        if (cudaMalloc(&b->park, bytes) != cudaSuccess)
        {
            cudaGetLastError();
            return B200CONV_OK;             /* no scratch: the one-CTA-per-frame kernel still works */
        }
        b->park_bytes   = bytes;
    }
    a.park          = b->park;
    return B200CONV_OK;
}

/* Reserves `count` consecutive slots of the job upload ring and returns their index. */
static int reserve_jobs(Batch *b, size_t count, cudaStream_t st, size_t *pos)
{
    if (count > b->job_cap)
        return fail(B200CONV_ERR_ARG, "job list too long (%zu)", count);
    if (b->job_pos + count > b->job_cap)
    {
        CU(cudaStreamSynchronize(st));      /* everything queued from the ring has been consumed */
        b->job_pos  = 0;
    }
    *pos        = b->job_pos;
    b->job_pos += count;
    return B200CONV_OK;
}

static int push_jobs(Batch *b, size_t pos, size_t count, cudaStream_t st)
{
    if (count == 0)
        return B200CONV_OK;
    CU(cudaMemcpyAsync(b->d_jobs + pos, b->h_jobs + pos, count * sizeof(Job), cudaMemcpyHostToDevice, st));
    return B200CONV_OK;
}

static StepArgs base_args(const Batch *b)
{
    StepArgs a;
    memset(&a, 0, sizeof(a));
    a.inst      = b->d_desc;
    a.active    = b->d_active;
    a.tw        = b->tw[b->rank];
    a.flags     = b->host_io ? uint32_t(STEP_HOST_IO) : 0u;
    a.ypart     = b->ypart;
    a.ring_head = b->d_ring_head;
    a.error     = b->h_error;       /* UVA: the mapped host word is addressable from the device */
    a.rank      = uint32_t(b->rank);
    a.n_active  = uint32_t(b->active.size());
    a.splits    = 1;
    return a;
}

static uint64_t algo_bytes(const Batch *b, const Instance &in, size_t qa, size_t qb)
{
    /* DESIGN.md: 16*F*bins + 24*F per instance-frame, bins = partitions of F taps in range */
    size_t lo   = (qa > in.q_lo) ? qa : in.q_lo;
    size_t hi   = (qb < in.q_lo + in.nq) ? qb : in.q_lo + in.nq;
    size_t rows = (hi > lo) ? hi - lo : 0;
    size_t bins = (rows > 0) ? rows - 1 : 0;
    (void)b;
    return uint64_t(16) * in.F * bins + uint64_t(24) * in.F;
}

/* ------------------------------------------------------------------------------------------- */
/* create / free                                                                                */

static int create_impl(b200conv_batch_t **out, int device, size_t instances)
{
    if ((out == nullptr) || (instances == 0) || (instances > (size_t(1) << 20)))
        return fail(B200CONV_ERR_ARG, "b200conv_create: bad arguments");
    *out = nullptr;

    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if ((e != cudaSuccess) || (count == 0))
        return fail(B200CONV_ERR_CUDA, "no CUDA device available (%s); this engine has no CPU fallback",
                    cudaGetErrorString(e));
    if (device < 0)
        CU(cudaGetDevice(&device));
    if (device >= count)
        return fail(B200CONV_ERR_ARG, "device %d out of range (%d devices)", device, count);

    Batch *b = new (std::nothrow) Batch();
    if (b == nullptr)
        return fail(B200CONV_ERR_NOMEM, "out of host memory");
    b->device   = device;
    b->n        = instances;
    b->inst.resize(instances);
    b->h_desc.resize(instances);
    b->h_ring_head.assign(instances, 0);
    b->h_slot_done.assign(FRAME_SLOTS * instances, 0);
    b->g_pos.assign(instances, 0);
    b->g_jobs.reserve(instances);
    b->g_fft.reserve(instances);
    b->g_mac.reserve(instances);
    b->g_part.reserve(instances);
    memset(b->h_desc.data(), 0, instances * sizeof(InstDesc));

    ENTER_DEVICE(b);
    int rc = B200CONV_OK;
    do
    {
        cudaDeviceProp prop;
        if (cudaGetDeviceProperties(&prop, device) == cudaSuccess)
            b->sm_count = prop.multiProcessorCount;
        #define CU_BRK(call) { cudaError_t e_ = (call); if (e_ != cudaSuccess) { rc = fail(B200CONV_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(e_)); break; } }
        CU_BRK(cudaStreamCreateWithFlags(&b->stream, cudaStreamNonBlocking));
        CU_BRK(cudaEventCreateWithFlags(&b->ev_done, cudaEventDisableTiming));
        CU_BRK(cudaEventCreateWithFlags(&b->ev_pend, cudaEventDisableTiming));
        CU_BRK(cudaEventCreateWithFlags(&b->ev_last, cudaEventDisableTiming));
        CU_BRK(cudaMalloc(&b->d_desc, instances * sizeof(InstDesc)));
        CU_BRK(cudaMalloc(&b->d_active, instances * sizeof(uint32_t)));
        b->job_cap = 64 * instances;
        if (b->job_cap < JOB_RING_MIN)  b->job_cap = JOB_RING_MIN;
        if (b->job_cap > JOB_RING_MAX)  b->job_cap = JOB_RING_MAX;
        if (b->job_cap < 3 * instances) b->job_cap = 3 * instances;    /* one unfused step: three lists */
        CU_BRK(cudaMallocHost(&b->h_jobs, b->job_cap * sizeof(Job)));
        CU_BRK(cudaMalloc(&b->d_jobs, b->job_cap * sizeof(Job)));
        CU_BRK(cudaMemset(b->d_desc, 0, instances * sizeof(InstDesc)));
        CU_BRK(cudaMalloc(&b->d_tickets, FRAME_SLOTS * instances * sizeof(uint32_t)));
        CU_BRK(cudaMemset(b->d_tickets, 0, FRAME_SLOTS * instances * sizeof(uint32_t)));
        CU_BRK(cudaMalloc(&b->d_slot_done, FRAME_SLOTS * instances * sizeof(uint32_t)));
        CU_BRK(cudaMemset(b->d_slot_done, 0, FRAME_SLOTS * instances * sizeof(uint32_t)));
        CU_BRK(cudaMalloc(&b->d_la_cnt, 2 * LA_BUFS * instances * sizeof(uint32_t)));
        CU_BRK(cudaMemset(b->d_la_cnt, 0, 2 * LA_BUFS * instances * sizeof(uint32_t)));
        CU_BRK(cudaHostAlloc(&b->h_error, 64, cudaHostAllocMapped | cudaHostAllocPortable));
        *b->h_error = 0;
        CU_BRK(cudaMalloc(&b->d_ring_head, (instances + 1) * sizeof(uint32_t)));       /* + the chain head (k_mac) */
        CU_BRK(cudaMemset(b->d_ring_head, 0, (instances + 1) * sizeof(uint32_t)));
        #undef CU_BRK
    } while (false);

    if (rc != B200CONV_OK)
    {
        std::string keep = g_last_error;
        b200conv_free(b);
        g_last_error = keep;
        return rc;
    }
    *out = b;
    return B200CONV_OK;
}

extern "C" void b200conv_free(b200conv_batch_t *b)
{
    if (b == nullptr)
        return;
    DeviceScope device_scope_(b->device);
    quiesce(b);
    for (Instance &in : b->inst)
        free_instance_buffers(in);
    for (float2 *t : b->tw)
        if (t) cudaFree(t);
    if (b->ypart)       cudaFree(b->ypart);
    if (b->park)        cudaFree(b->park);
    if (b->d_partials)  cudaFree(b->d_partials);
    if (b->init_scratch) cudaFree(b->init_scratch);
    for (int i = 0; i < 2; ++i)
    {
        if (b->init_stage[i])   cudaFreeHost(b->init_stage[i]);
        if (b->init_ev[i])      cudaEventDestroy(b->init_ev[i]);
    }
    if (b->d_desc)      cudaFree(b->d_desc);
    if (b->d_active)    cudaFree(b->d_active);
    if (b->d_tickets)   cudaFree(b->d_tickets);
    if (b->d_slot_done) cudaFree(b->d_slot_done);
    if (b->d_la_cnt)    cudaFree(b->d_la_cnt);
    if (b->la_T)        cudaFree(b->la_T);
    if (b->d_ring_head) cudaFree(b->d_ring_head);
    if (b->h_error)     cudaFreeHost(b->h_error);
    if (b->d_jobs)      cudaFree(b->d_jobs);
    if (b->h_jobs)      cudaFreeHost(b->h_jobs);
    if (b->h_in)        cudaFreeHost(b->h_in);
    if (b->h_out)       cudaFreeHost(b->h_out);
    if (b->d_in)        cudaFree(b->d_in);
    if (b->d_out)       cudaFree(b->d_out);
    b200conv_reduce_disconnect(b);
    if (b->ev_done)     cudaEventDestroy(b->ev_done);
    if (b->ev_pend)     cudaEventDestroy(b->ev_pend);
    if (b->ev_last)     cudaEventDestroy(b->ev_last);
    for (cudaEvent_t ev : b->prof_events)
        cudaEventDestroy(ev);
    if (b->stream)      cudaStreamDestroy(b->stream);
    delete b;
}

/* ------------------------------------------------------------------------------------------- */
/* init / destroy                                                                               */

extern "C" int b200conv_destroy(b200conv_batch_t *b, size_t idx)
{
    if ((b == nullptr) || (idx >= b->n))
        return fail(B200CONV_ERR_ARG, "b200conv_destroy: bad handle or index");
    Instance &in = b->inst[idx];
    if (!in.active)
        return B200CONV_OK;
    if (in.g_sharers > 0)
        return fail(B200CONV_ERR_STATE, "instance %zu lends its IR spectra to %zu other instance(s): destroy those first",
                    idx, in.g_sharers);
    ENTER_DEVICE(b);
    CU(quiesce(b));
    if (in.g_owner >= 0)
        b->inst[size_t(in.g_owner)].g_sharers -= 1;
    free_instance_buffers(in);
    in = Instance();
    rebuild_tables(b);
    return B200CONV_OK;
}

/* Convolver::init for MANY instances at once (Convolver.cpp:77-215 per instance):
 *   - ONE device allocation (slab) holds the IR spectra, the input-spectrum ring and the frame
 *     buffers of all of them, allocated before any old state is touched (:103-108);
 *   - the impulse responses go up through a double-buffered page-locked staging area, the copy of
 *     chunk k + 1 into it overlapping the transfer of chunk k;
 *   - ONE transform launch covers every partition of every instance (the per-partition
 *     fastconv_parse of :183-197), one more forms the folded spectra and keeps taps [0, F).
 * counts[i] == 0 destroys instance idx[i] (:80-84). */
static const size_t INIT_STAGE_FLOATS  = size_t(4) << 20;      /* 16 MiB per page-locked staging buffer */
static const size_t INIT_CHUNK_FLOATS  = size_t(16) << 20;     /* padded IR samples transformed per round: 64 MiB of taps,
                                                                   128 MiB of spectra -- bounded scratch, whatever the job */
static const size_t INIT_KEEP_BYTES    = size_t(64) << 20;     /* device scratch up to this size stays with the batch */
static const int    INIT_COPY_THREADS  = 4;                    /* host threads filling one staging buffer */

static void slab_release(Slab *s)
{
    if ((s != nullptr) && (--s->refs == 0))
    {
        cudaFree(s->base);
        delete s;
    }
}

/* pageable -> page-locked copy, split over a few host threads above 1 MiB (one core moves ~8 GB/s,
 * less than PCIe 5 takes) */
static void staged_copy(float *dst, const float *src, size_t n)
{
    if (n < (size_t(1) << 18))
    {
        memcpy(dst, src, n * sizeof(float));
        return;
    }
    std::thread pool[INIT_COPY_THREADS - 1];
    const size_t per = (n + INIT_COPY_THREADS - 1) / INIT_COPY_THREADS;
    for (int t = 1; t < INIT_COPY_THREADS; ++t)
    {
        const size_t lo = (per * t < n) ? per * t : n, hi = (lo + per < n) ? lo + per : n;
        pool[t - 1]     = std::thread([=]() { if (hi > lo) memcpy(dst + lo, src + lo, (hi - lo) * sizeof(float)); });
    }
    memcpy(dst, src, ((per < n) ? per : n) * sizeof(float));
    for (int t = 1; t < INIT_COPY_THREADS; ++t)
        pool[t - 1].join();
}

static int init_many_impl(b200conv_batch_t *b, size_t count, const size_t *idx, const float *const *data,
                          const size_t *counts, size_t rank, const float *phases, const size_t *part_offsets)
{
    if ((b == nullptr) || (count == 0) || (idx == nullptr) || (data == nullptr) || (counts == nullptr))
        return fail(B200CONV_ERR_ARG, "b200conv_init_many: bad arguments");

    /* Convolver.cpp:87 : clamp through a signed value */
    long r = long(rank);
    if (r < B200CONV_RANK_MIN) r = B200CONV_RANK_MIN;
    if (r > B200CONV_RANK_MAX) r = B200CONV_RANK_MAX;
    rank = size_t(r);
    const size_t F      = size_t(1) << (rank - 1);

    std::vector<char> touched(b->n, 0);
    size_t live = 0, rows_total = 0, slab_floats = 0, rows_max = 0;
    for (size_t k = 0; k < count; ++k)
    {
        if ((idx[k] >= b->n) || touched[idx[k]])
            return fail(B200CONV_ERR_ARG, "b200conv_init_many: index %zu out of range or repeated", idx[k]);
        touched[idx[k]]     = 1;
        if (b->inst[idx[k]].g_sharers > 0)
            return fail(B200CONV_ERR_STATE, "instance %zu lends its IR spectra to %zu other instance(s): destroy those first",
                        idx[k], b->inst[idx[k]].g_sharers);
        if (counts[k] == 0)
            continue;
        if (data[k] == nullptr)
            return fail(B200CONV_ERR_ARG, "b200conv_init: NULL impulse response");
        const size_t po     = (part_offsets != nullptr) ? part_offsets[k] : 0;
        const size_t bins   = (counts[k] + F - 1) >> (rank - 1);    /* Convolver.cpp:93 */
        if ((po + bins + 1) >= (size_t(1) << 31))
            return fail(B200CONV_ERR_ARG, "impulse response too long");
        ++live;
        rows_total         += bins;
        rows_max            = (bins > rows_max) ? bins : rows_max;
        /* G: bins + 1 rows | ring: S rows (float2 [F]) | aux: 3 F floats */
        slab_floats        += 2 * F * (bins + 1) + 2 * F * (po + bins + 1 + RING_SPARE) + 3 * F;
    }
    for (size_t i = 0; i < b->n; ++i)
        if ((!touched[i]) && b->inst[i].active && (live > 0) && (b->inst[i].rank != rank))
            return fail(B200CONV_ERR_ARG, "all instances of a batch share one rank (%zu active, %zu requested)",
                        b->inst[i].rank, rank);

    ENTER_DEVICE(b);
    CU(quiesce(b));                 /* the tables and buffers below may be in use by queued launches */
    cudaStream_t st = b->stream;

    if (live == 0)
    {
        for (size_t k = 0; k < count; ++k)
            TRY(b200conv_destroy(b, idx[k]));
        return B200CONV_OK;
    }
    if (b->tw[rank] == nullptr)
        TRY(make_twiddles(uint32_t(rank), &b->tw[rank]));

    const bool trace = (getenv("B200CONV_INIT_TRACE") != nullptr);
    auto now_ms = []() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    const double t_start = now_ms();

    /* Scratch, bounded whatever the job: the instances are transformed in rounds of whole instances
     * whose padded IRs fit INIT_CHUNK_FLOATS (a single longer IR gets a round of its own). */
    size_t chunk_rows   = INIT_CHUNK_FLOATS / F;
    if (chunk_rows < rows_max)      chunk_rows = rows_max;
    if (chunk_rows > rows_total)    chunk_rows = rows_total;
    const size_t stage_floats   = (rows_total * F < INIT_STAGE_FLOATS) ? rows_total * F : INIT_STAGE_FLOATS;
    const size_t scratch_bytes  = chunk_rows * F * (sizeof(float) + sizeof(float2)) + live * sizeof(FoldDesc) + 256;

    /* Allocate everything new before touching the old state (Convolver.cpp:103-108). */
    float *slab_mem = nullptr;
    cudaError_t e = cudaMalloc(&slab_mem, slab_floats * sizeof(float));
    if ((e == cudaSuccess) && (scratch_bytes > b->init_scratch_bytes))
    {
        if (b->init_scratch) cudaFree(b->init_scratch);
        b->init_scratch         = nullptr;
        b->init_scratch_bytes   = 0;
        e = cudaMalloc(&b->init_scratch, scratch_bytes);
        if (e == cudaSuccess)
            b->init_scratch_bytes   = scratch_bytes;
    }
    if ((e == cudaSuccess) && (stage_floats > b->init_stage_floats))
    {
        for (int i = 0; i < 2; ++i)
        {
            if (b->init_stage[i]) cudaFreeHost(b->init_stage[i]);
            b->init_stage[i]        = nullptr;
        }
        b->init_stage_floats    = 0;
        for (int i = 0; (i < 2) && (e == cudaSuccess); ++i)
            e = cudaMallocHost(&b->init_stage[i], stage_floats * sizeof(float));
        if (e == cudaSuccess)
            b->init_stage_floats    = stage_floats;
    }
    for (int i = 0; (i < 2) && (e == cudaSuccess); ++i)
        if (b->init_ev[i] == nullptr)
            e = cudaEventCreateWithFlags(&b->init_ev[i], cudaEventDisableTiming);
    if (e != cudaSuccess)
    {
        if (slab_mem) cudaFree(slab_mem);
        cudaGetLastError();
        return fail(B200CONV_ERR_NOMEM, "allocation failed for %zu impulse response(s): %s", live, cudaGetErrorString(e));
    }
    float *irdev        = reinterpret_cast<float *>(b->init_scratch);
    float2 *H           = reinterpret_cast<float2 *>(irdev + chunk_rows * F);
    FoldDesc *d_fold    = reinterpret_cast<FoldDesc *>(reinterpret_cast<unsigned char *>(H + chunk_rows * F) + 128);
    Slab *slab          = new Slab();
    slab->base          = slab_mem;
    slab->refs          = live;
    const double t_alloc = now_ms();

    /* carve the slab: all IR spectra first, then ring + frame buffers (one memset clears those) */
    std::vector<FoldDesc> fold(live);
    std::vector<Instance> fresh(live);
    std::vector<size_t> which_k(live);
    size_t at = 0, slot = 0;
    for (size_t k = 0; k < count; ++k)
    {
        if (counts[k] == 0) continue;
        fresh[slot].G   = reinterpret_cast<float2 *>(slab_mem + at);
        at             += 2 * F * (((counts[k] + F - 1) >> (rank - 1)) + 1);
        which_k[slot]   = k;
        ++slot;
    }
    const size_t clear_from = at;
    slot = 0;
    for (size_t k = 0; k < count; ++k)
    {
        if (counts[k] == 0) continue;
        const size_t po     = (part_offsets != nullptr) ? part_offsets[k] : 0;
        const size_t bins   = (counts[k] + F - 1) >> (rank - 1);
        Instance &in        = fresh[slot];
        in.ring             = reinterpret_cast<float2 *>(slab_mem + at);
        at                 += 2 * F * (po + bins + 1 + RING_SPARE);
        in.aux              = slab_mem + at;
        at                 += 3 * F;
        in.slab             = slab;
        in.active           = true;
        in.conv_size        = counts[k];
        in.rank             = rank;
        in.F                = F;
        in.bins             = bins;
        in.nq               = bins + 1;                     /* folded overlap: one extra row */
        in.q_lo             = po;
        in.S                = po + bins + 1 + RING_SPARE;
        float fo            = ((phases != nullptr) ? phases[k] : 0.0f) * float(F);     /* Convolver.cpp:140, fp32 */
        in.off              = ((fo > 0.0f) && (fo < 1.8e19f)) ? (size_t(fo) % F) : 0;
        in.off0             = in.off;
        fold[slot].G        = in.G;
        fold[slot].head     = (po == 0) ? in.aux + 2 * F : nullptr;
        fold[slot].h_row    = 0;                            /* within its round, set below */
        fold[slot].bins     = uint32_t(bins);
        fold[slot].pad      = 0;
        ++slot;
    }

    int rc = B200CONV_OK;
    double t_upload = 0.0;
    do
    {
        #define CU_BRK(call) { cudaError_t e_ = (call); if (e_ != cudaSuccess) { rc = fail(B200CONV_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(e_)); break; } }
        CU_BRK(cudaMemsetAsync(slab_mem + clear_from, 0, (slab_floats - clear_from) * sizeof(float), st));

        int which = 0;
        bool used[2] = { false, false };
        for (size_t s0 = 0; (s0 < live) && (rc == B200CONV_OK); )
        {
            /* one round: instances s0 .. s1-1 */
            size_t s1 = s0, rows = 0;
            while ((s1 < live) && ((s1 == s0) || (rows + fold[s1].bins <= chunk_rows)))
            {
                fold[s1].h_row  = rows;
                rows           += fold[s1].bins;
                ++s1;
            }
            const double t_round = now_ms();
            CU_BRK(cudaMemsetAsync(irdev, 0, rows * F * sizeof(float), st));    /* the zero padding of every last partition */
            CU_BRK(cudaMemcpyAsync(d_fold, fold.data() + s0, (s1 - s0) * sizeof(FoldDesc), cudaMemcpyHostToDevice, st));

            /* upload: host -> staging buffer (CPU copy, a few threads) -> device (DMA), two buffers in flight */
            for (size_t sl = s0; (sl < s1) && (rc == B200CONV_OK); ++sl)
            {
                const size_t k  = which_k[sl];
                for (size_t done = 0; done < counts[k]; )
                {
                    size_t c    = counts[k] - done;
                    if (c > b->init_stage_floats)   c = b->init_stage_floats;
                    if (used[which])
                        CU_BRK(cudaEventSynchronize(b->init_ev[which]));
                    staged_copy(b->init_stage[which], data[k] + done, c);
                    CU_BRK(cudaMemcpyAsync(irdev + fold[sl].h_row * F + done, b->init_stage[which], c * sizeof(float),
                                           cudaMemcpyHostToDevice, st));
                    CU_BRK(cudaEventRecord(b->init_ev[which], st));
                    used[which] = true;
                    which      ^= 1;
                    done       += c;
                }
                b->stats.h2d_bytes += counts[k] * sizeof(float);
            }
            if (rc != B200CONV_OK) break;
            t_upload   += now_ms() - t_round;

            /* H_p = spectrum of taps [pF, (p+1)F) zero padded -- the per-partition fastconv_parse of
             * Convolver.cpp:183-197 for every partition of every instance of the round, one launch */
            StepArgs a  = base_args(b);
            a.rank      = uint32_t(rank);
            a.tw        = b->tw[rank];
            a.jobs      = nullptr;
            a.flags     = STEP_LINEAR_JOBS;
            a.src       = irdev;
            a.dst       = reinterpret_cast<float *>(H);
            CU_BRK(launch_fwd(a, uint32_t(rows), st));
            b->stats.launches++;

            size_t max_bins = 0;
            for (size_t sl = s0; sl < s1; ++sl)
                max_bins    = (fold[sl].bins > max_bins) ? fold[sl].bins : max_bins;
            dim3 grid(uint32_t((F + 255) / 256), uint32_t((max_bins + 1 < 1024) ? max_bins + 1 : 1024),
                      uint32_t((s1 - s0 < 64) ? s1 - s0 : 64));
            k_fold_many<<<grid, 256, 0, st>>>(d_fold, uint32_t(s1 - s0), H, irdev, uint32_t(F));
            CU_BRK(cudaGetLastError());
            b->stats.launches++;
            s0          = s1;
        }
        if (rc != B200CONV_OK) break;
        CU_BRK(cudaStreamSynchronize(st));
        #undef CU_BRK
    } while (false);

    const double t_done = now_ms();
    if (b->init_scratch_bytes > INIT_KEEP_BYTES)
    {
        /* a big job's scratch goes back; small ones (a plugin re-loading its IR) keep theirs */
        cudaStreamSynchronize(st);
        cudaFree(b->init_scratch);
        b->init_scratch         = nullptr;
        b->init_scratch_bytes   = 0;
    }
    if (rc != B200CONV_OK)
    {
        cudaStreamSynchronize(st);
        cudaFree(slab_mem);
        delete slab;
        return rc;
    }
    if (trace)
        fprintf(stderr, "b200conv_init_many: %zu instances, %.1f MB of taps: alloc %.2f ms, upload (enqueue) %.2f ms, "
                        "all rounds + drain %.2f ms, release %.2f ms\n", live, rows_total * F * 4e-6,
                t_alloc - t_start, t_upload, t_done - t_alloc, now_ms() - t_done);

    /* swap in (Convolver.cpp:108-142) */
    slot = 0;
    for (size_t k = 0; k < count; ++k)
    {
        Instance &in    = b->inst[idx[k]];
        if (in.g_owner >= 0)
            b->inst[size_t(in.g_owner)].g_sharers -= 1;
        free_instance_buffers(in);
        in              = (counts[k] == 0) ? Instance() : fresh[slot++];
    }
    rebuild_tables(b);
    return B200CONV_OK;
}

static int init_range_impl(b200conv_batch_t *b, size_t idx, const float *data, size_t count,
                           size_t rank, float phase, size_t part_offset)
{
    if ((b == nullptr) || (idx >= b->n))
        return fail(B200CONV_ERR_ARG, "b200conv_init: bad handle or index");
    if (count == 0)                                         /* Convolver.cpp:80-84 */
        return b200conv_destroy(b, idx);
    return init_many_impl(b, 1, &idx, &data, &count, rank, &phase, &part_offset);
}

extern "C" int b200conv_init(b200conv_batch_t *b, size_t idx, const float *data, size_t count,
                             size_t rank, float phase)
{
    return b200conv_init_range(b, idx, data, count, rank, phase, 0);
}

/* Convolver::init for instance `idx` with the SAME impulse response (and rank) as the initialised
 * instance `src_idx`: the device spectra are shared, only the input-spectrum ring and the frame
 * buffers are new.  Many channels through one reverb pay for one set of IR spectra. */
static int init_shared_impl(b200conv_batch_t *b, size_t idx, size_t src_idx, float phase)
{
    if ((b == nullptr) || (idx >= b->n) || (src_idx >= b->n) || (idx == src_idx))
        return fail(B200CONV_ERR_ARG, "b200conv_init_shared: bad handle or index");
    const Instance &from = b->inst[(b->inst[src_idx].g_owner >= 0) ? size_t(b->inst[src_idx].g_owner) : src_idx];
    const size_t owner = size_t(&from - b->inst.data());
    if ((!from.active) || (owner == idx))
        return fail(B200CONV_ERR_STATE, "b200conv_init_shared: instance %zu is not initialised", src_idx);
    if (b->inst[idx].g_sharers > 0)
        return fail(B200CONV_ERR_STATE, "instance %zu lends its IR spectra to other instances: destroy those first", idx);

    ENTER_DEVICE(b);
    CU(quiesce(b));
    cudaStream_t st = b->stream;
    const size_t F  = from.F;

    Instance fresh;
    cudaError_t e   = cudaMalloc(&fresh.ring, from.S * F * sizeof(float2));
    if (e == cudaSuccess) e = cudaMalloc(&fresh.aux, 3 * F * sizeof(float));
    if (e != cudaSuccess)
    {
        if (fresh.ring) cudaFree(fresh.ring);
        cudaGetLastError();
        return fail(B200CONV_ERR_NOMEM, "device allocation failed: %s", cudaGetErrorString(e));
    }
    e = cudaMemsetAsync(fresh.ring, 0, from.S * F * sizeof(float2), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(fresh.aux, 0, 2 * F * sizeof(float), st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(fresh.aux + 2 * F, from.aux + 2 * F, F * sizeof(float), cudaMemcpyDeviceToDevice, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess)
    {
        cudaFree(fresh.ring);
        cudaFree(fresh.aux);
        return fail(B200CONV_ERR_CUDA, "b200conv_init_shared: %s", cudaGetErrorString(e));
    }

    Instance &in    = b->inst[idx];
    if (in.g_owner >= 0)
        b->inst[size_t(in.g_owner)].g_sharers -= 1;
    free_instance_buffers(in);
    in              = fresh;
    in.G            = from.G;
    in.g_owner      = long(owner);
    in.g_sharers    = 0;
    b->inst[owner].g_sharers += 1;
    in.active       = true;
    in.conv_size    = from.conv_size;
    in.rank         = from.rank;
    in.F            = F;
    in.bins         = from.bins;
    in.nq           = from.nq;
    in.q_lo         = from.q_lo;
    in.S            = from.S;
    float fo        = phase * float(F);                     /* Convolver.cpp:140, fp32 */
    in.off          = ((fo > 0.0f) && (fo < 1.8e19f)) ? (size_t(fo) % F) : 0;
    in.off0         = in.off;
    in.frames       = 0;
    in.pend_valid   = false;
    rebuild_tables(b);
    return B200CONV_OK;
}

/* ------------------------------------------------------------------------------------------- */
/* process                                                                                      */

/* All active instances sit on a frame boundary and `frames` whole frames arrive: derive the
 * jobs on the device, three launches per frame for all instances x partitions. */
static bool eager_possible(const Batch *b)
{
    return (b->opt_eager != 0) && (b->opt_fused != 0) && (b->rank >= 8) && (b->rank <= 11) &&
           (b->reduce.mode == 0) && (!b->profiling) && (!b->active.empty());
}

static int process_uniform(Batch *b, float *dst, size_t dst_stride, const float *src, size_t stride,
                           size_t frames, cudaStream_t st)
{
    const uint32_t nact = uint32_t(b->active.size());
    if (b->uniform_stale)
        b->desc_dirty   = true;         /* the general path moved the frame counters one by one */
    b->uniform_stale = false;
    const bool tables_changed = b->desc_dirty;
    TRY(upload_tables(b, st));
    MacPlan plan    = plan_mac(uint32_t(b->rank), nact, uint32_t(b->max_nq), b->sm_count,
                               b->tune_splits, b->tune_stages);
    const size_t F  = size_t(1) << (b->rank - 1);
    const bool eager = b->eager_call && (frames == 1) && eager_possible(b);
    /* one extra row per job when the pending MAC runs ahead (it must not be re-allocated between
     * the pending launch and the call that consumes it) */
    TRY(ensure_ypart(b, size_t(nact) * (plan.splits + 1) * F * sizeof(float2), st));
    if (tables_changed || (b->pend_splits != plan.splits))
        b->pend_ready   = false;

    uint64_t per_frame_bytes = 0;
    for (uint32_t i : b->active)
        per_frame_bytes += algo_bytes(b, b->inst[i], 0, size_t(-1));

    StepArgs a      = base_args(b);
    a.src           = src;
    a.dst           = dst;
    a.stride        = stride;
    a.stride_dst    = dst_stride;
    a.splits        = plan.splits;
    a.n_jobs        = nact;
    a.t_base        = b->t_batch;
    const bool fused = (b->opt_fused != 0) && (b->rank <= 13);     /* k_frame: ranks 8..13 */
    if ((b->reduce.mode != 0) && (!fused))
        return fail(B200CONV_ERR_STATE, "the fused cross-GPU reduce needs the one-launch-per-block path (ranks 8..13, fused = 1)");
    plan.sh.bias    = fused ? uint32_t(b->opt_bias) : 0;
    bool used_multi = false;
    for (size_t f = 0; f < frames; )
    {
        a.frame0        = uint32_t(f);
        a.n_jobs        = nact;
        /* several whole frames in one call: transform them all, then ONE pass over the IR
         * spectra serves tf frames (k_mac_multi), then all inverse transforms */
        uint32_t tf     = 0;
        for (uint32_t c = (b->reduce.mode != 0) ? 0u : uint32_t(b->opt_multi); c >= 2; c >>= 1)
            if (frames - f >= c) { tf = c; break; }
        if (tf >= 2)
        {
            MacPlan mp      = plan;
            mp.sh.bias      = 0;
            /* the register window limits occupancy (8 frames: 1 CTA/SM, 4: 2, 2: 3), so the
             * bytes in flight come from a deeper shared-memory ring instead */
            mp.sh.NS        = (tf == 8) ? 8 : (tf == 4) ? 6 : 4;
            mp.smem         = size_t(2) * mp.sh.NS * mp.sh.QB * mp.sh.TB * sizeof(float2) + 2 * mp.sh.NS * sizeof(uint64_t) + 16;
            TRY(ensure_ypart(b, size_t(nact) * tf * mp.splits * F * sizeof(float2), st));
            hist_reset(st, b->device);
            a.ypart         = b->ypart;
            a.n_jobs        = nact * tf;
            CU(launch_fwd(a, nact * tf, st));
            CU(launch_mac_multi(a, mp, nact, tf, st));
            TRY(attach_park(b, a, size_t(nact) * tf, st));
            CU(launch_inv(a, nact * tf, st));
            hist_unknown(st, b->device);
            b->chain_valid  = false;
            b->ahead_valid  = false;
            b->la_live      = false;
            b->stats.launches       += 3;
            b->stats.mac_launches   += 1;
            b->stats.mac_algo_bytes += per_frame_bytes * tf;
            b->stats.mac_stream_bytes += per_frame_bytes * tf;
            b->stats.frames         += uint64_t(nact) * tf;
            used_multi      = true;
            b->pend_ready   = false;
            f              += tf;
            continue;
        }
        if (fused && (!used_multi))
        {
            /* Lookahead (kernels.cuh, LA_BUFS): a stream of one-frame calls in uniform mode.  Chosen from
             * the call pattern and the batch's shape only -- never from pdl, profiling, the stream or the
             * early-read options -- so that every way of running a stream sums in the same order.  A
             * synchronous call, a multi-frame call, the general path or any table change ends the schedule;
             * the next one starts with a priming group (full sums, tails for the group after it). */
            uint32_t K      = 0;
            if ((frames == 1) && (!b->eager_call) && (b->reduce.mode == 0))
                K               = lookahead_k(b, per_frame_bytes);
            uint64_t launch_bytes = per_frame_bytes;
            a.la_K          = 0;
            if (K != 0)
            {
                const uint64_t t    = a.t_base + f;
                if ((!b->la_live) || (b->la_K != K) || (b->la_splits != plan.splits) || (b->la_nact != nact) ||
                    tables_changed || (b->la_next_t != t))
                {
                    TRY(ensure_la(b, size_t(LA_BUFS) * nact * K * plan.splits * F * sizeof(float2), st));
                    b->la_origin    = t;
                }
                const uint64_t rel  = t - b->la_origin;
                const uint32_t g    = uint32_t((rel / K) % LA_BUFS);
                a.la_T          = b->la_T;
                a.la_prod       = b->d_la_cnt;
                a.la_cons       = b->d_la_cnt + LA_BUFS * b->n;
                a.la_K          = K;
                a.la_c          = uint32_t(rel % K);
                a.la_use        = (rel >= K) ? 1u : 0u;
                a.la_get        = g;
                a.la_put        = (g + 1) % LA_BUFS;
                a.la_put_need   = b->la_cons_cnt[a.la_put];
                a.la_get_need   = b->la_prod_cnt[a.la_get];
                if (a.la_use)
                    b->la_cons_cnt[a.la_get] += 1;
                b->la_prod_cnt[a.la_put] += plan.splits * plan.tiles;
                b->la_live      = true;
                b->la_K         = K;
                b->la_splits    = plan.splits;
                b->la_nact      = nact;
                b->la_next_t    = t + 1;
                launch_bytes    = 0;
                for (uint32_t i : b->active)
                    launch_bytes   += la_stream_bytes(b->inst[i], K, a.la_use != 0, plan.sh, plan.splits);
            }
            else
                b->la_live      = false;
            /* one launch per block for all instances x partitions.  May its input transform run
             * ahead of the launches still in flight on this stream? (FrameHistory) */
            bool early = false, serial = false, dst_clash = false;
            {
                /* worth it only while the transform is a visible share of the block: a launch that
                 * streams for tens of microseconds hides the chain anyway */
                const bool capable = (b->opt_pdl != 0) && (!b->profiling) && (launch_bytes <= EARLY_MAX_BYTES) &&
                                     ((b->opt_early_src == 2) || ((b->opt_early_src == 1) && (st == b->stream)));
                const BlockRows in  = { reinterpret_cast<uintptr_t>(src + f * F), stride * sizeof(float), F * sizeof(float), b->n };
                const BlockRows out = { reinterpret_cast<uintptr_t>(dst + f * F), dst_stride * sizeof(float), F * sizeof(float), b->n };
                hist_launch(st, b->device, capable, in, out, &early, &serial, &dst_clash);
            }
            a.flags        &= ~uint32_t(STEP_EARLY_SRC | STEP_ORDER_DST);
            if (early)
                a.flags        |= STEP_EARLY_SRC;
            if (dst_clash)
                a.flags        |= STEP_ORDER_DST;  /* e.g. a cascade re-using one hand-over block: the tail of the
                                                      next launch must not overwrite what a launch in flight reads */
            /* pipelined tails (FRAME_SLOTS in kernels.cuh): this launch's rows, tickets and sequence number */
            a.seq           = b->frame_seq;
            a.n_cap         = uint32_t(b->n);
            a.slot_done     = ((b->opt_pdl != 0) && (!b->profiling)) ? b->d_slot_done : nullptr;
            a.ypart         = ypart_slot(b, a.seq);
            if (a.slot_done != nullptr)
                b->frame_seq   += 1;            /* only pipelined launches take part in the slot rotation */
            if (eager && b->pend_ready && (b->pend_t == b->t_batch + f) && (!tables_changed) && (b->pend_seq == a.seq))
            {
                /* partitions q >= 1 were summed ahead of time (launch_pending_mac): transform the
                 * input, add partition 0, invert -- one CTA per instance */
                MacPlan fp      = plan;
                fp.splits       = 1;
                fp.sh.bias      = 0;
                StepArgs af     = a;
                af.splits       = 1;
                af.rows         = b->pend_splits + 1;
                af.row0         = b->pend_splits;
                af.sum0         = b->pend_splits - 1;       /* the pending MAC folded its rows into this one */
                af.flags       |= STEP_HEAD_ONLY;
                /* A synchronous host call on the own stream: every launch that delivered an earlier
                 * block has completed (the caller has its output), and the predecessor in the
                 * stream is this batch's pending MAC, which never touches the caller's input block
                 * -- the block is fetched and transformed under that MAC whatever the launch size. */
                if ((st == b->stream) && (b->opt_pdl != 0) && (b->opt_early_src != 0))
                    af.flags       |= STEP_EARLY_SRC;
                CU(launch_mac(b, af, fp, nact, st, true, serial));
            }
            else
                CU(launch_mac(b, a, plan, nact, st, true, serial));
            b->pend_ready   = false;
            b->last_was_frame = (st == b->stream) && (!b->profiling);
            b->stats.launches       += 1;
            b->stats.mac_stream_bytes += launch_bytes;
        }
        else
        {
            MacPlan sp      = plan;
            sp.sh.bias      = 0;
            b->pend_ready   = false;
            b->la_live      = false;
            b->stats.mac_stream_bytes += per_frame_bytes;
            const bool ahead = (b->rank >= 14) && (b->opt_pdl != 0) && (!b->profiling) && (b->opt_chain_ahead != 0) && (frames == 1);
            if (ahead)
            {
                /* Block-by-block callers at ranks 14..16: partitions q >= 1 of block t need complete frames
                 * only, so their MAC is launched one block AHEAD -- behind the inverse transform of block
                 * t - 1 -- into a row slot of its own, and streams under that inverse transform and under
                 * the transform of block t; partition 0 is added by the inverse transform of block t
                 * (STEP_Q0_IN_INV).  Stream order per call:  k_fwd(t)  k_inv(t)  k_mac(t + 1).
                 * What orders them: chain_head ("frames < x are final", published by k_inv(t) once
                 * k_fwd(t) has completed; k_mac(t + 1) polls it), row slots t mod FRAME_SLOTS, and one
                 * CTA of every kernel that waits for the launch before it as its last instruction. */
                const uint64_t t    = a.t_base + a.frame0;
                const uint32_t t32  = uint32_t(t);
                uint32_t *head      = b->d_ring_head + b->n;
                auto mac_ahead = [&](uint64_t t_of, bool pdl) -> cudaError_t
                {
                    StepArgs am     = a;
                    am.t_base       = t_of - a.frame0;
                    am.ypart        = ypart_slot(b, uint32_t(t_of));
                    am.flags       |= STEP_FROM_Q1 | STEP_AHEAD;
                    am.chain_head   = head;
                    return launch_mac(b, am, sp, nact, st, false, false, pdl);
                };
                if (!(b->ahead_valid && (b->ahead_t == t) && (b->ahead_splits == sp.splits)))
                {
                    /* cold start (or a MAC launched ahead for a block that never came): seed the chain head by
                     * a copy and launch this block's MAC without the attribute -- both full dependencies */
                    CU(cudaMemcpyAsync(head, &t32, sizeof(t32), cudaMemcpyHostToDevice, st));
                    CU(mac_ahead(t, false));
                    b->stats.launches += 1;
                }
                bool early = false, serial = false, dst_clash = false;
                {
                    const bool capable = (b->opt_early_src == 2) || ((b->opt_early_src == 1) && (st == b->stream));
                    const BlockRows in  = { reinterpret_cast<uintptr_t>(src + f * F), stride * sizeof(float), F * sizeof(float), b->n };
                    const BlockRows out = { reinterpret_cast<uintptr_t>(dst + f * F), dst_stride * sizeof(float), F * sizeof(float), b->n };
                    hist_launch(st, b->device, capable, in, out, &early, &serial, &dst_clash);
                }
                StepArgs ai     = a;
                ai.ypart        = ypart_slot(b, t32);
                TRY(attach_park(b, ai, nact, st));      /* (may synchronise) */
                StepArgs af     = a;
                if (early)
                    af.flags       |= STEP_EARLY_SRC;
                CU(launch_fwd(af, nact, st, !serial));
                ai.flags       |= STEP_Q0_IN_INV;
                ai.chain_head   = head;
                CU(launch_inv(ai, nact, st, true, b->d_tickets));
                CU(mac_ahead(t + 1, true));
                b->ahead_valid  = true;
                b->ahead_t      = t + 1;
                b->ahead_splits = sp.splits;
                b->chain_valid  = true;
                b->chain_next   = t32 + 1u;
                b->stats.launches       += 3;
                b->stats.mac_launches   += 1;
                b->stats.mac_algo_bytes += per_frame_bytes;
                b->stats.frames         += nact;
                f              += 1;
                continue;
            }
            b->ahead_valid  = false;
            hist_reset(st, b->device);
            /* Ranks 14..16: the three kernels of a block are chained with programmatic serialisation --
             * the partition stream of q >= 1 runs beside the block's own transform (which only the
             * stage with q = 0 needs, taken last, STEP_AFTER_FWD), table staging overlaps the launch
             * before; every kernel orders itself with griddepcontrol.wait. */
            const bool chain = (b->rank >= 14) && (b->opt_pdl != 0) && (!b->profiling);
            TRY(attach_park(b, a, nact, st));       /* (may synchronise: before the chain starts) */
            CU(launch_fwd(a, nact, st, chain));
            StepArgs am     = a;
            if (chain)
                am.flags       |= STEP_AFTER_FWD;
            {
                /* "the spectra of all frames < t are final": published by the k_mac of block t - 1; whenever
                 * that was not the launch before this one (first block, a multi-frame pass, the general
                 * path, another frame counter) the word is seeded by a copy -- a full dependency */
                const uint32_t t32 = uint32_t(a.t_base + a.frame0);
                if ((!b->chain_valid) || (b->chain_next != t32))
                    CU(cudaMemcpyAsync(b->d_ring_head + b->n, &t32, sizeof(t32), cudaMemcpyHostToDevice, st));
                am.chain_head   = b->d_ring_head + b->n;
                b->chain_valid  = true;
                b->chain_next   = t32 + 1u;
            }
            CU(launch_mac(b, am, sp, nact, st, false, false, chain));
            CU(launch_inv(a, nact, st, chain, b->d_tickets));      /* nact <= instances counters */
            hist_unknown(st, b->device);
            b->stats.launches       += 3;
        }
        b->stats.mac_launches   += 1;
        b->stats.mac_algo_bytes += per_frame_bytes;
        b->stats.frames         += nact;
        f              += 1;
    }
    if (used_multi)
        b->desc_dirty   = true;     /* ring_head was bypassed: re-seed before the next k_frame */
    b->t_batch     += frames;
    for (uint32_t i : b->active)
    {
        b->inst[i].frames      += frames;
        b->inst[i].pend_valid   = false;
    }
    return B200CONV_OK;
}

/* Sums, ahead of time, the partitions q >= 1 of the block that the next whole-frame call will
 * bring (they need complete frames only): rows 0 .. splits-1 of every job; row `splits` is left
 * for that call's own partition 0.  Called by the synchronous host entry points after the
 * output of the current block is on its way, so the work hides behind the host's round trip --
 * the GPU analogue of the reference spreading its tail blocks over the frame
 * (Convolver.cpp:199-210,275). */
static int launch_pending_mac(Batch *b, cudaStream_t st)
{
    if (!eager_possible(b) || b->desc_dirty)
        return B200CONV_OK;
    for (uint32_t i : b->active)
        if (b->inst[i].off != 0)
            return B200CONV_OK;

    const uint32_t nact = uint32_t(b->active.size());
    MacPlan plan    = plan_mac(uint32_t(b->rank), nact, uint32_t(b->max_nq), b->sm_count,
                               b->tune_splits, b->tune_stages);
    const size_t F  = size_t(1) << (b->rank - 1);
    if (size_t(nact) * (plan.splits + 1) * F * sizeof(float2) > b->ypart_slot_bytes)
        return B200CONV_OK;                 /* sized by the next process call */

    StepArgs a      = base_args(b);
    a.ypart         = ypart_slot(b, b->frame_seq);      /* the slot of the k_frame launch that will add partition 0 */
    b->pend_seq     = b->frame_seq;
    a.splits        = plan.splits;
    a.rows          = plan.splits + 1;
    a.row0          = 0;
    a.flags        |= STEP_FROM_Q1;
    a.fold_tickets  = b->d_tickets + size_t(b->frame_seq % uint32_t(FRAME_SLOTS)) * b->n;   /* the slot's: idle until that launch */
    a.n_jobs        = nact;
    a.t_base        = b->t_batch;           /* the block about to arrive */
    a.frame0        = 0;
    plan.sh.bias    = 0;
    /* Behind a k_frame launch of this batch the MAC may start early: it polls ring_head for the
     * spectrum that launch publishes and holds its rows back until that launch has completed. */
    /* auto: early only while the caller keeps the GPU busy (the previous pending MAC was still
     * running when this call arrived); a caller that comes back once per audio block gets the
     * delivering launch to itself */
    const bool early = (b->opt_pdl != 0) && b->last_was_frame &&
                       ((b->opt_early_pend == 2) || ((b->opt_early_pend == 1) && b->caller_busy));
    if (early)
        a.flags        |= STEP_WAIT_HEAD;
    CU(launch_mac_raw(a, plan, nact, st, early));
    b->last_was_frame = false;
    b->stats.launches       += 1;
    b->stats.mac_launches   += 1;
    b->pend_ready   = true;
    b->pend_t       = b->t_batch;
    b->pend_splits  = plan.splits;
    return B200CONV_OK;
}

static inline uint32_t slot_of(const Instance &in, uint64_t t)
{
    uint64_t tm = t % in.S;
    return uint32_t((tm == 0) ? 0 : in.S - tm);
}

/* Where the kernels of one step find its job list: up to JOB_PACK jobs ride in the kernel's
 * parameter space (*dev = NULL: no copy operation in the stream -- a real-time call is one kernel
 * launch); longer lists are uploaded from the page-locked ring. */
static int publish_jobs(Batch *b, const Job *list, size_t count, cudaStream_t st, JobPack *pack, const Job **dev)
{
    if (count <= JOB_PACK)
    {
        memcpy(pack->j, list, count * sizeof(Job));
        *dev        = nullptr;
        return B200CONV_OK;
    }
    size_t at   = 0;
    TRY(reserve_jobs(b, count, st, &at));
    memcpy(b->h_jobs + at, list, count * sizeof(Job));
    TRY(push_jobs(b, at, count, st));
    *dev        = b->d_jobs + at;
    return B200CONV_OK;
}

/* Any call size / any phase, ranks 8..13: ONE launch per step.  Every instance contributes at most
 * one job, and a job is whatever the instance needs next, in this order (kernels.cuh, Job):
 *     P1   samples that continue the frame in progress, answered from its pending block
 *     FFT  the frame is complete: its spectrum enters the ring
 *     MAC  what the complete frames contribute to the frame about to start (q >= 1) -> the new
 *          pending block; or, for a whole frame taken from the input on a frame boundary, every
 *          partition -> the output block
 *     P2   the first samples of that new frame, answered from the block just computed
 * A 256-sample call of a phase-shifted instance (BASELINE config 2) is P1 + FFT + MAC + P2 in one
 * k_frame<GEN> launch; a call inside a frame is one k_partial_fused launch. */
static int process_general_fused(Batch *b, float *dst, size_t dst_stride, const float *src, size_t stride,
                                 size_t count, cudaStream_t st)
{
    const size_t F      = size_t(1) << (b->rank - 1);
    TRY(upload_tables(b, st));
    hist_reset(st, b->device);          /* every CTA of the job-list form waits for all earlier launches */
    b->la_live          = false;        /* a lookahead schedule restarts with a priming group */
    std::vector<size_t> &pos = b->g_pos;
    std::vector<Job> &jobs = b->g_jobs;
    for (uint32_t i : b->active)
        pos[i]          = 0;

    for (;;)
    {
        jobs.clear();
        uint64_t bytes  = 0;
        size_t n_mac = 0, n_fft = 0, max_nq = 0;
        for (uint32_t i : b->active)
        {
            Instance &in = b->inst[i];
            if (pos[i] >= count)
                continue;
            float *cur  = in.aux, *pend = in.aux + F;
            const float *x  = src + size_t(i) * stride;
            float *y        = dst + size_t(i) * dst_stride;
            size_t rem  = count - pos[i];
            Job j;
            memset(&j, 0, sizeof(j));
            j.inst      = i;

            auto pending_mac = [&]()
            {
                /* what the complete frames contribute to frame t = in.frames: partitions q >= 1 */
                j.flags    |= JOB_MAC;
                j.dst       = pend;
                j.slot0     = slot_of(in, in.frames);
                j.tlo       = uint32_t(in.frames);
                j.qa        = uint32_t((in.q_lo > 1) ? in.q_lo : 1);
                j.qb        = uint32_t(in.q_lo + in.nq);
                bytes      += algo_bytes(b, in, j.qa, j.qb);
                in.pend_valid = true;
                b->stats.frames += 1;
            };

            if ((in.off == 0) && (rem >= F))
            {
                /* a whole frame on a frame boundary: FFT -> every partition -> IFFT -> out */
                j.flags     = JOB_FFT | JOB_MAC;
                j.src       = x + pos[i];
                j.dst       = y + pos[i];
                j.slot0     = slot_of(in, in.frames);
                j.spec      = in.ring + size_t(j.slot0) * F;
                j.tlo       = uint32_t(in.frames);
                j.qa        = uint32_t(in.q_lo);
                j.qb        = uint32_t(in.q_lo + in.nq);
                bytes      += algo_bytes(b, in, j.qa, j.qb);
                in.frames  += 1;
                in.pend_valid = false;
                b->stats.frames += 1;
                pos[i]     += F;
            }
            else if (!in.pend_valid)
            {
                /* the pending block of the frame in progress first; its samples ride along (P2)
                 * unless they would complete the frame -- that is the next step's P1 + FFT */
                pending_mac();
                if (rem < F - in.off)
                {
                    size_t n2   = (rem < PART_MAX) ? rem : PART_MAX;
                    j.psrc2     = x + pos[i];
                    j.pdst2     = y + pos[i];
                    j.off2      = uint32_t(in.off);
                    j.n2        = uint32_t(n2);
                    in.off     += n2;
                    pos[i]     += n2;
                }
            }
            else
            {
                size_t n1   = (rem < F - in.off) ? rem : F - in.off;
                if (n1 > PART_MAX)
                    n1          = PART_MAX;
                j.psrc      = x + pos[i];
                j.pdst      = y + pos[i];
                j.off       = uint32_t(in.off);
                j.n         = uint32_t(n1);
                in.off     += n1;
                pos[i]     += n1;
                rem        -= n1;
                if (in.off == F)
                {
                    /* the frame is complete: its spectrum enters the ring in this same launch */
                    j.flags    |= JOB_FFT | JOB_FFT_PREV;
                    j.src       = cur;
                    j.spec      = in.ring + size_t(slot_of(in, in.frames)) * F;
                    in.frames  += 1;
                    in.off      = 0;
                    in.pend_valid = false;
                    j.tlo       = uint32_t(in.frames);      /* = t of the frame about to start */
                    if (rem < F)
                    {
                        /* ... and so does what the samples after it will need */
                        pending_mac();
                        size_t n2   = (rem < PART_MAX) ? rem : PART_MAX;
                        if (n2 > 0)
                        {
                            j.psrc2     = x + pos[i];
                            j.pdst2     = y + pos[i];
                            j.off2      = 0;
                            j.n2        = uint32_t(n2);
                            in.off      = n2;
                            pos[i]     += n2;
                        }
                    }
                }
            }
            if (j.flags & JOB_MAC)
            {
                ++n_mac;
                if (in.nq > max_nq)
                    max_nq      = in.nq;
            }
            if (j.flags & JOB_FFT)
                ++n_fft;
            jobs.push_back(j);
        }
        if (jobs.empty())
            break;

        StepArgs a  = base_args(b);
        JobPack pack;
        TRY(publish_jobs(b, jobs.data(), jobs.size(), st, &pack, &a.jobs));
        a.n_jobs    = uint32_t(jobs.size());
        if ((n_mac == 0) && (n_fft == 0))
        {
            /* every job sits inside a frame: store + answer, one CTA per job */
            k_partial_fused<<<a.n_jobs, 256, 0, st>>>(a, pack);
            CU(cudaGetLastError());
            b->stats.launches += 1;
            continue;
        }
        MacPlan plan = plan_mac(uint32_t(b->rank), uint32_t(jobs.size()), uint32_t((max_nq > 0) ? max_nq : 2),
                                b->sm_count, b->tune_splits, b->tune_stages);
        plan.sh.bias = 0;
        /* one more row per job: the direct-form answers that the job's CTAs share out (k_frame_gen) */
        TRY(ensure_ypart(b, jobs.size() * (plan.splits + 1) * F * sizeof(float2), st));
        a.ypart     = b->ypart;
        a.splits    = plan.splits;
        CU(launch_frame_gen(a, plan, a.n_jobs, b->d_tickets, pack, (b->opt_pdl != 0) && (!b->profiling), st));
        b->stats.launches       += 1;
        if (n_mac > 0)
        {
            b->stats.mac_launches   += 1;
            b->stats.mac_algo_bytes += bytes;
            b->stats.mac_stream_bytes += bytes;
        }
    }

    hist_unknown(st, b->device);
    b->chain_valid = false;
    b->ahead_valid = false;
    b->uniform_stale = true;    /* per-instance frame counters moved independently of t_batch */
    b->pend_ready = false;
    return B200CONV_OK;
}

/* The same schedule with one kernel per stage (ranks 14..16, whose frame transform does not fit a
 * k_frame CTA, and fused = 0):
 *     k_store + k_partial (samples of frames in progress, answered from their pending block)
 *  -> k_fwd               (frames that just completed, and whole frames taken from the input)
 *  -> k_mac -> k_inv      (whole frames: every partition -> output;
 *                          frames about to start: partitions q >= 1 -> their pending block)
 * and each instance contributes at most one item per stage. */
static int process_general_staged(Batch *b, float *dst, size_t dst_stride, const float *src, size_t stride,
                                  size_t count, cudaStream_t st)
{
    const size_t F      = size_t(1) << (b->rank - 1);
    TRY(upload_tables(b, st));
    hist_reset(st, b->device);
    std::vector<size_t> &pos = b->g_pos;
    std::vector<Job> &fft = b->g_fft, &mac = b->g_mac, &part = b->g_part;
    for (uint32_t i : b->active)
        pos[i]          = 0;

    for (;;)
    {
        fft.clear(); mac.clear(); part.clear();
        uint64_t bytes = 0;
        for (uint32_t i : b->active)
        {
            Instance &in = b->inst[i];
            if (pos[i] >= count)
                continue;
            float *cur  = in.aux, *pend = in.aux + F;
            Job j;

            auto push_frame_spectrum = [&](const float *samples)
            {
                memset(&j, 0, sizeof(j));
                j.inst      = i;
                j.src       = samples;
                j.slot0     = slot_of(in, in.frames);
                j.spec      = in.ring + size_t(j.slot0) * F;
                fft.push_back(j);
            };
            auto push_pending_block = [&]()
            {
                /* what the complete frames contribute to the frame about to start: q >= 1 */
                memset(&j, 0, sizeof(j));
                j.inst      = i;
                j.dst       = pend;
                j.slot0     = slot_of(in, in.frames);
                j.qa        = uint32_t((in.q_lo > 1) ? in.q_lo : 1);
                j.qb        = uint32_t(in.q_lo + in.nq);
                mac.push_back(j);
                bytes      += algo_bytes(b, in, j.qa, j.qb);
                in.pend_valid = true;
                b->stats.frames += 1;
            };

            size_t rem  = count - pos[i];
            if (!((in.off == 0) && (rem >= F)))
            {
                if (!in.pend_valid)
                {
                    /* the pending block first; the samples are answered in the next step */
                    push_pending_block();
                    continue;
                }

                /* the next samples of the frame in progress (zero latency for any call size) */
                size_t n    = (rem < F - in.off) ? rem : F - in.off;
                memset(&j, 0, sizeof(j));
                j.inst      = i;
                j.psrc      = src + size_t(i) * stride + pos[i];
                j.pdst      = dst + size_t(i) * dst_stride + pos[i];
                j.off       = uint32_t(in.off);
                j.n         = uint32_t(n);
                part.push_back(j);
                in.off     += n;
                pos[i]     += n;
                rem        -= n;
                if (in.off < F)
                    continue;                       /* frame still open: the call is exhausted */

                /* the frame is complete: spectrum into the ring in this same step (k_store runs
                 * before k_fwd), and straight on to what the next samples will need */
                push_frame_spectrum(cur);
                in.frames  += 1;
                in.off      = 0;
                in.pend_valid = false;
                if (rem < F)
                {
                    push_pending_block();
                    continue;
                }
            }

            /* a whole frame at once: FFT -> MAC over every partition -> IFFT -> out */
            push_frame_spectrum(src + size_t(i) * stride + pos[i]);
            j.dst       = dst + size_t(i) * dst_stride + pos[i];
            j.qa        = uint32_t(in.q_lo);
            j.qb        = uint32_t(in.q_lo + in.nq);
            fft.back()  = j;
            mac.push_back(j);
            bytes      += algo_bytes(b, in, j.qa, j.qb);
            in.frames  += 1;
            in.pend_valid = false;
            b->stats.frames += 1;
            pos[i]     += F;
        }

        size_t total = fft.size() + mac.size() + part.size();
        if (total == 0)
            break;

        /* the transform / MAC lists are uploaded (their kernels take device lists); a short list of
         * samples to answer rides in the launch parameters */
        size_t maxn = 0;
        for (const Job &pj : part)
            if (pj.n > maxn) maxn = pj.n;
        const bool part_packed = (!part.empty()) && (maxn <= 256) && (part.size() <= JOB_PACK);
        const size_t n_up = (part_packed ? 0 : part.size()) + fft.size() + mac.size();
        const size_t part_up = part_packed ? 0 : part.size();
        size_t at = 0;
        if (n_up > 0)
        {
            TRY(reserve_jobs(b, n_up, st, &at));
            Job *hj = b->h_jobs + at;
            if (part_up > 0)    memcpy(hj, part.data(), part.size() * sizeof(Job));
            if (!fft.empty())   memcpy(hj + part_up, fft.data(), fft.size() * sizeof(Job));
            if (!mac.empty())   memcpy(hj + part_up + fft.size(), mac.data(), mac.size() * sizeof(Job));
            TRY(push_jobs(b, at, n_up, st));
        }
        const Job *dj = b->d_jobs + at;

        StepArgs a  = base_args(b);
        if (!part.empty())
        {
            a.jobs      = part_packed ? nullptr : dj;
            a.n_jobs    = uint32_t(part.size());
            size_t deepest = 0;
            for (const Job &pj : part)
                if (size_t(pj.off) + pj.n > deepest) deepest = size_t(pj.off) + pj.n;
            const uint32_t max_tiles = uint32_t((F + PO_TILE - 1) / PO_TILE);
            if ((maxn <= PT_MAXN) && (deepest > 2 * PO_TILE) && (a.n_jobs <= 65535u))
            {
                /* deep inside a long frame: the tap tiles of every job side by side */
                if (part.size() > b->partials_jobs)
                {
                    CU(cudaStreamSynchronize(st));
                    if (b->d_partials) cudaFree(b->d_partials);
                    b->d_partials       = nullptr;
                    b->partials_jobs    = 0;
                    size_t want         = (part.size() < 16) ? 16 : part.size();    /* outside the steady state only */
                    CU(cudaMalloc(&b->d_partials, want * max_tiles * PT_MAXN * sizeof(double)));
                    b->partials_jobs    = want;
                }
                JobPack pack;
                if (part_packed)
                    memcpy(pack.j, part.data(), part.size() * sizeof(Job));
                dim3 gt(uint32_t((deepest - 1) / PO_TILE + 1), a.n_jobs);
                k_partial_tiles<<<gt, 256, 0, st>>>(a, pack, b->d_partials, b->d_tickets, max_tiles);
                CU(cudaGetLastError());
                b->stats.launches += 1;
            }
            else if (maxn <= 256)
            {
                JobPack pack;
                if (part_packed)
                    memcpy(pack.j, part.data(), part.size() * sizeof(Job));
                k_partial_fused<<<a.n_jobs, 256, 0, st>>>(a, pack);
                CU(cudaGetLastError());
                b->stats.launches += 1;
            }
            else
            {
                /* long segments: store, then share each job's outputs among several CTAs */
                dim3 gs(uint32_t((maxn + 255) / 256), (a.n_jobs < 65535u) ? a.n_jobs : 65535u);
                k_store<<<gs, 256, 0, st>>>(a);
                CU(cudaGetLastError());
                dim3 gp(uint32_t((maxn + 31) / 32 > 64 ? 64 : (maxn + 31) / 32), gs.y);
                k_partial<<<gp, 256, 0, st>>>(a);
                CU(cudaGetLastError());
                b->stats.launches += 2;
            }
        }
        if (!fft.empty())
        {
            a.jobs      = dj + part_up;
            a.n_jobs    = uint32_t(fft.size());
            CU(launch_fwd(a, a.n_jobs, st));
            b->stats.launches++;
        }
        if (!mac.empty())
        {
            MacPlan plan = plan_mac(uint32_t(b->rank), uint32_t(mac.size()), uint32_t(b->max_nq),
                                    b->sm_count, b->tune_splits, b->tune_stages);
            TRY(ensure_ypart(b, mac.size() * plan.splits * F * sizeof(float2), st));
            a.ypart     = b->ypart;
            a.jobs      = dj + part_up + fft.size();
            a.n_jobs    = uint32_t(mac.size());
            a.splits    = plan.splits;
            CU(launch_mac(b, a, plan, a.n_jobs, st));
            TRY(attach_park(b, a, a.n_jobs, st));
            CU(launch_inv(a, a.n_jobs, st));
            b->stats.launches       += 2;
            b->stats.mac_launches   += 1;
            b->stats.mac_algo_bytes += bytes;
            b->stats.mac_stream_bytes += bytes;
        }
    }

    /* ring_head was bypassed and the per-instance frame counters moved: both matter only to a
     * k_frame launch, which refreshes the tables first (uniform_stale) */
    hist_unknown(st, b->device);
    b->chain_valid = false;
    b->ahead_valid = false;
    b->uniform_stale = true;
    b->pend_ready = false;
    return B200CONV_OK;
}

static int process_general(Batch *b, float *dst, size_t dst_stride, const float *src, size_t stride,
                           size_t count, cudaStream_t st)
{
    if ((b->opt_fused != 0) && (b->rank <= 13))
        return process_general_fused(b, dst, dst_stride, src, stride, count, st);
    return process_general_staged(b, dst, dst_stride, src, stride, count, st);
}

static int process_device2_impl(b200conv_batch_t *b, float *dst, size_t dst_stride,
                                        const float *src, size_t src_stride, size_t count, void *stream)
{
    if (b == nullptr)
        return fail(B200CONV_ERR_ARG, "b200conv_process_device: NULL handle");
    if (count == 0)
        return B200CONV_OK;
    if ((dst == nullptr) || (src == nullptr) || ((b->n > 1) && ((src_stride < count) || (dst_stride < count))))
        return fail(B200CONV_ERR_ARG, "b200conv_process_device: bad buffers");
    ENTER_DEVICE(b);
    cudaStream_t st = (stream != nullptr) ? cudaStream_t(stream) : b->stream;
    TRY(check_device_error(b));
    b->last_was_frame = false;
    if (b->eager_call)
    {
        b->caller_busy  = b->pend_inflight && (cudaEventQuery(b->ev_pend) == cudaErrorNotReady);
        cudaGetLastError();         /* "not ready" is an answer, not an error: do not leave it behind
                                       for the cudaGetLastError() after the next <<< >>> launch */
    }
    if (b->pend_inflight && (st != b->stream))
        CU(cudaStreamWaitEvent(st, b->ev_pend, 0));     /* a pending MAC may still be running on the own stream */

    /* not initialised -> zeros (Convolver.cpp:219-223) */
    if (b->active.size() < b->n)
        hist_reset(st, b->device);
    for (size_t i = 0; i < b->n; )
    {
        if (b->inst[i].active) { ++i; continue; }
        size_t j = i;
        while ((j < b->n) && (!b->inst[j].active))
            ++j;
        if ((j - i == 1) || (dst_stride == count))
            CU(cudaMemsetAsync(dst + i * dst_stride, 0, ((j - i - 1) * dst_stride + count) * sizeof(float), st));
        else
            CU(cudaMemset2DAsync(dst + i * dst_stride, dst_stride * sizeof(float), 0, count * sizeof(float), j - i, st));
        i = j;
    }
    if (b->active.empty())
        return B200CONV_OK;

    const size_t F = size_t(1) << (b->rank - 1);
    bool uniform = (count % F) == 0;
    for (uint32_t i : b->active)
        if (b->inst[i].off != 0)
            uniform = false;

    int rc;
    if (uniform)
        rc = process_uniform(b, dst, dst_stride, src, src_stride, count / F, st);
    else if (b->reduce.mode != 0)
        return fail(B200CONV_ERR_STATE, "the fused cross-GPU reduce handles whole-frame calls only");
    else
        rc = process_general(b, dst, dst_stride, src, src_stride, count, st);
    if ((rc == B200CONV_OK) && (st != b->stream))
    {
        CU(cudaEventRecord(b->ev_last, st));
        b->last_foreign = true;
    }
    return rc;
}

extern "C" int b200conv_process_device(b200conv_batch_t *b, float *dst, const float *src,
                                       size_t stride, size_t count, void *stream)
{
    return b200conv_process_device2(b, dst, stride, src, stride, count, stream);
}

/* End of a synchronous host call: the output of this block is on its way on the own stream.
 * Queue the next block's pending MAC behind it, but return as soon as the OUTPUT is complete. */
static int finish_sync_call(Batch *b)
{
    CU(cudaEventRecord(b->ev_done, b->stream));
    TRY(launch_pending_mac(b, b->stream));
    if (b->pend_ready)
    {
        CU(cudaEventRecord(b->ev_pend, b->stream));
        b->pend_inflight = true;
    }
    CU(cudaEventSynchronize(b->ev_done));
    hist_reset(b->stream, b->device);   /* every launch that delivered this block has completed */
    return check_device_error(b);
}

static int ensure_staging(Batch *b, size_t floats)
{
    if (floats <= b->stage_floats)
        return B200CONV_OK;
    CU(cudaStreamSynchronize(b->stream));
    if (b->h_in)  cudaFreeHost(b->h_in);
    if (b->h_out) cudaFreeHost(b->h_out);
    if (b->d_in)  cudaFree(b->d_in);
    if (b->d_out) cudaFree(b->d_out);
    b->h_in = b->h_out = b->d_in = b->d_out = nullptr;
    b->stage_floats = 0;
    CU(cudaMallocHost(&b->h_in, floats * sizeof(float)));
    CU(cudaMallocHost(&b->h_out, floats * sizeof(float)));
    CU(cudaHostGetDevicePointer(&b->h_in_dev, b->h_in, 0));
    CU(cudaHostGetDevicePointer(&b->h_out_dev, b->h_out, 0));
    CU(cudaMalloc(&b->d_in, floats * sizeof(float)));
    CU(cudaMalloc(&b->d_out, floats * sizeof(float)));
    b->stage_floats = floats;
    return B200CONV_OK;
}

extern "C" int b200conv_process(b200conv_batch_t *b, float *const *dst, const float *const *src,
                                size_t count)
{
    if (b == nullptr)
        return fail(B200CONV_ERR_ARG, "b200conv_process: NULL handle");
    if (count == 0)
        return B200CONV_OK;
    if ((dst == nullptr) || (src == nullptr))
        return fail(B200CONV_ERR_ARG, "b200conv_process: NULL buffer table");
    for (size_t i = 0; i < b->n; ++i)
        if ((dst[i] == nullptr) || (src[i] == nullptr))
            return fail(B200CONV_ERR_ARG, "b200conv_process: NULL buffer for instance %zu", i);
    ENTER_DEVICE(b);

    /* samples per instance per pass: bounded staging, at least one frame */
    size_t cap = (size_t(1) << 24) / b->n;
    if (cap > 65536)    cap = 65536;
    size_t F   = (b->rank > 0) ? (size_t(1) << (b->rank - 1)) : 128;
    if (cap < F)        cap = F;
    cap        = (cap / F) * F;

    for (size_t done = 0; done < count; )
    {
        size_t c = count - done;
        if (c > cap)
            c = cap;
        TRY(ensure_staging(b, b->n * c));
        for (size_t i = 0; i < b->n; ++i)
            if (b->inst[i].active)
                memcpy(b->h_in + i * c, src[i] + done, c * sizeof(float));
        /* the gathered block sits in page-locked memory: short blocks are read and written by the
         * kernels in place across PCIe (no copy operations in the stream), long ones are copied */
        const bool in_place = (b->opt_zero_copy != 0) && (b->n * c * sizeof(float) <= (size_t(4) << 20));
        b->eager_call = true;
        int rc;
        if (in_place)
        {
            b->host_io      = true;
            rc              = b200conv_process_device(b, b->h_out_dev, b->h_in_dev, c, c, b->stream);
            b->host_io      = false;
        }
        else
        {
            hist_reset(b->stream, b->device);
            CU(cudaMemcpyAsync(b->d_in, b->h_in, b->n * c * sizeof(float), cudaMemcpyHostToDevice, b->stream));
            rc              = b200conv_process_device(b, b->d_out, b->d_in, c, c, b->stream);
        }
        b->eager_call = false;
        TRY(rc);
        if (!in_place)
            CU(cudaMemcpyAsync(b->h_out, b->d_out, b->n * c * sizeof(float), cudaMemcpyDeviceToHost, b->stream));
        if (done + c >= count)
            TRY(finish_sync_call(b));
        else
            CU(cudaStreamSynchronize(b->stream));
        for (size_t i = 0; i < b->n; ++i)
            memcpy(dst[i] + done, b->h_out + i * c, c * sizeof(float));
        b->stats.h2d_bytes += b->n * c * sizeof(float);
        b->stats.d2h_bytes += b->n * c * sizeof(float);
        done += c;
    }
    return B200CONV_OK;
}

extern "C" int b200conv_process_planar(b200conv_batch_t *b, float *dst, const float *src,
                                       size_t stride, size_t count)
{
    if (b == nullptr)
        return fail(B200CONV_ERR_ARG, "b200conv_process_planar: NULL handle");
    if (count == 0)
        return B200CONV_OK;
    if ((dst == nullptr) || (src == nullptr) || (stride < count))
        return fail(B200CONV_ERR_ARG, "b200conv_process_planar: bad buffers");
    ENTER_DEVICE(b);

    /* Page-locked host matrices are mapped into the device address space (UVA): the kernels
     * read the input block and write the output block across PCIe themselves -- the input fetch
     * hides under the first partition stages, and two copy operations (and their launch
     * latencies) disappear from the call. */
    if (b->opt_zero_copy)
    {
        cudaPointerAttributes as, ad;
        if ((cudaPointerGetAttributes(&as, src) == cudaSuccess) && (cudaPointerGetAttributes(&ad, dst) == cudaSuccess) &&
            (as.type == cudaMemoryTypeHost) && (ad.type == cudaMemoryTypeHost) &&
            (as.devicePointer != nullptr) && (ad.devicePointer != nullptr))
        {
            b->eager_call = true;
            b->host_io    = true;
            int rc = b200conv_process_device(b, static_cast<float *>(ad.devicePointer),
                                             static_cast<const float *>(as.devicePointer), stride, count, b->stream);
            b->eager_call = false;
            b->host_io    = false;
            TRY(rc);
            TRY(finish_sync_call(b));
            b->stats.h2d_bytes += b->n * count * sizeof(float);
            b->stats.d2h_bytes += b->n * count * sizeof(float);
            return B200CONV_OK;
        }
        cudaGetLastError();     /* pageable memory: not an error, take the staged path */
    }

    size_t cap = (size_t(1) << 24) / b->n;
    if (cap > 65536)    cap = 65536;
    size_t F   = (b->rank > 0) ? (size_t(1) << (b->rank - 1)) : 128;
    if (cap < F)        cap = F;
    cap        = (cap / F) * F;

    for (size_t done = 0; done < count; )
    {
        size_t c = count - done;
        if (c > cap)
            c = cap;
        TRY(ensure_staging(b, b->n * c));
        hist_reset(b->stream, b->device);
        CU(cudaMemcpy2DAsync(b->d_in, c * sizeof(float), src + done, stride * sizeof(float),
                             c * sizeof(float), b->n, cudaMemcpyHostToDevice, b->stream));
        b->eager_call = true;
        int rc = b200conv_process_device(b, b->d_out, b->d_in, c, c, b->stream);
        b->eager_call = false;
        TRY(rc);
        CU(cudaMemcpy2DAsync(dst + done, stride * sizeof(float), b->d_out, c * sizeof(float),
                             c * sizeof(float), b->n, cudaMemcpyDeviceToHost, b->stream));
        if (done + c >= count)
            TRY(finish_sync_call(b));
        else
            CU(cudaStreamSynchronize(b->stream));
        b->stats.h2d_bytes += b->n * c * sizeof(float);
        b->stats.d2h_bytes += b->n * c * sizeof(float);
        done += c;
    }
    return B200CONV_OK;
}

extern "C" int b200conv_sync(b200conv_batch_t *b)
{
    if (b == nullptr)
        return fail(B200CONV_ERR_ARG, "b200conv_sync: NULL handle");
    ENTER_DEVICE(b);
    CU(quiesce(b));
    return check_device_error(b);
}

/* ------------------------------------------------------------------------------------------- */
/* queries                                                                                      */

extern "C" size_t b200conv_data_size(const b200conv_batch_t *b, size_t idx)
{
    return ((b != nullptr) && (idx < b->n)) ? b->inst[idx].conv_size : 0;
}

extern "C" size_t b200conv_rank(const b200conv_batch_t *b, size_t idx)
{
    return ((b != nullptr) && (idx < b->n)) ? b->inst[idx].rank : 0;
}

extern "C" size_t b200conv_instances(const b200conv_batch_t *b)
{
    return (b != nullptr) ? b->n : 0;
}

extern "C" int b200conv_get_state(const b200conv_batch_t *b, size_t idx, b200conv_state_t *st)
{
    if ((b == nullptr) || (idx >= b->n) || (st == nullptr))
        return fail(B200CONV_ERR_ARG, "b200conv_get_state: bad arguments");
    const Instance &in = b->inst[idx];
    st->conv_size   = in.conv_size;
    st->rank        = in.rank;
    st->frame_size  = in.F;
    st->frame_off   = (in.off == in.F) ? 0 : in.off;    /* a complete frame rolls over lazily */
    st->bins        = in.bins;
    st->partitions  = in.nq;
    st->part_offset = in.q_lo;
    st->frames      = in.frames + ((in.active && (in.off == in.F)) ? 1 : 0);
    return B200CONV_OK;
}

extern "C" int b200conv_get_dump(const b200conv_batch_t *b, size_t idx, b200conv_dump_t *out)
{
    if ((b == nullptr) || (idx >= b->n) || (out == nullptr))
        return fail(B200CONV_ERR_ARG, "b200conv_get_dump: bad arguments");
    memset(out, 0, sizeof(*out));
    const Instance &in = b->inst[idx];
    if (!in.active)
        return B200CONV_OK;                                 /* construct(): everything NULL / 0 */

    const size_t F      = in.F, count = in.conv_size;
    out->vDataBuffer    = in.aux + F;
    out->vFrame         = in.aux;
    out->vConvBuffer    = b->ypart;
    out->vTaskData      = in.ring;
    out->vConvData      = in.G;
    out->vDirectData    = in.aux + 2 * F;
    out->vData          = in.G;
    out->nDataBufferSize = (in.bins + 1) * F;               /* Convolver.cpp:137 */
    out->nFrameSize     = F;
    out->nFrameOff      = (in.off == F) ? 0 : in.off;
    out->nDirectSize    = (count < 128) ? count : 128;      /* :141 */
    out->nConvSize      = count;
    out->nRank          = in.rank;

    /* the reference's partition map (:152-197): 128 direct taps, raising levels of 128, 256, ...
     * taps up to F / 2, then blocks of F */
    size_t left         = count - out->nDirectSize;
    size_t levels       = 0;
    for (size_t brank = 8; (left > 0) && (brank < in.rank); ++brank)
    {
        size_t n            = size_t(1) << (brank - 1);
        left               -= (left < n) ? left : n;
        ++levels;
    }
    out->nLevels        = levels;
    out->nBlocks        = (left + F - 1) / F;

    /* load spreading (:199-210), fp32 like the reference */
    const long steps    = long(F >> 7);
    if (steps <= 1)
    {
        out->nBlkInit       = out->nBlocks;
        out->fBlkCoef       = 0.0f;
    }
    else
    {
        out->nBlkInit       = 1;
        out->fBlkCoef       = (float(out->nBlocks) + 1e-3f) / (float(steps) - 1.0f);
    }

    /* nBlocksDone: nBlocks after init (:198); reset at the first sample of a frame (:268-272) and
     * raised at every 128-sample boundary that has received a sample (:275-285) */
    const size_t off    = out->nFrameOff;
    const bool rolled   = (in.off == F);                    /* complete frame, not rolled over here yet */
    const uint64_t done = in.frames + (rolled ? 1 : 0);     /* frames completed since init */
    const bool reset_seen = (in.off0 == 0) ? ((done > 0) || (off > 0))
                                           : ((done >= 2) || ((done == 1) && (off > 0)));
    if ((out->nBlocks == 0) || (!reset_seen) || (off == 0))
        out->nBlocksDone    = out->nBlocks;
    else
    {
        const size_t sub_id = (off - 1) >> 7;
        size_t target       = size_t(float(out->nBlkInit) + out->fBlkCoef * float(sub_id));
        out->nBlocksDone    = (target < out->nBlocks) ? target : out->nBlocks;
    }
    return B200CONV_OK;
}

extern "C" int b200conv_get_stats(const b200conv_batch_t *b, b200conv_stats_t *st)
{
    if ((b == nullptr) || (st == nullptr))
        return fail(B200CONV_ERR_ARG, "b200conv_get_stats: bad arguments");
    *st = b->stats;
    return B200CONV_OK;
}

extern "C" int b200conv_reset_stats(b200conv_batch_t *b)
{
    if (b == nullptr)
        return fail(B200CONV_ERR_ARG, "b200conv_reset_stats: NULL handle");
    memset(&b->stats, 0, sizeof(b->stats));
    return B200CONV_OK;
}

extern "C" int b200conv_set_profiling(b200conv_batch_t *b, int enable)
{
    if (b == nullptr)
        return fail(B200CONV_ERR_ARG, "b200conv_set_profiling: NULL handle");
    b->profiling    = (enable != 0);
    b->desc_dirty   = true;     /* profiled launches are not pipelined: the slot counters are re-seeded */
    b->pend_ready   = false;
    return B200CONV_OK;
}

extern "C" int b200conv_get_profile(b200conv_batch_t *b, double *mac_ms, uint64_t *mac_launches)
{
    if (b == nullptr)
        return fail(B200CONV_ERR_ARG, "b200conv_get_profile: NULL handle");
    ENTER_DEVICE(b);
    double total = 0.0;
    for (size_t i = 0; i + 1 < b->prof_used; i += 2)
    {
        CU(cudaEventSynchronize(b->prof_events[i + 1]));
        float ms = 0.0f;
        CU(cudaEventElapsedTime(&ms, b->prof_events[i], b->prof_events[i + 1]));
        total += ms;
    }
    if (mac_ms != nullptr)          *mac_ms = total;
    if (mac_launches != nullptr)    *mac_launches = b->prof_used / 2;
    b->prof_used = 0;
    return B200CONV_OK;
}

extern "C" void *b200conv_stream(b200conv_batch_t *b)
{
    return (b != nullptr) ? (void *)b->stream : nullptr;
}

extern "C" int b200conv_set_option(b200conv_batch_t *b, const char *name, int value)
{
    if ((b == nullptr) || (name == nullptr))
        return fail(B200CONV_ERR_ARG, "b200conv_set_option: bad arguments");
    if (!strcmp(name, "mac_splits") && (value >= 0) && (value <= 32))       b->tune_splits = value;
    else if (!strcmp(name, "chain_ahead") && (value >= 0) && (value <= 1)) { b->opt_chain_ahead = value; b->ahead_valid = false; }
    else if (!strcmp(name, "mac_tile") && ((value == 0) || (value == 256) || (value == 512) || (value == 1024))) g_tune_tile = value;
    else if (!strcmp(name, "mac_stages") && ((value == 0) || ((value >= 2) && (value <= 12)))) b->tune_stages = value;
    else if (!strcmp(name, "fused") && (value >= 0) && (value <= 1))        b->opt_fused = value;
    else if (!strcmp(name, "fft_bias") && (value >= 0) && (value <= 64))    b->opt_bias = value;
    else if (!strcmp(name, "pdl") && (value >= 0) && (value <= 1))          b->opt_pdl = value;
    else if (!strcmp(name, "zero_copy") && (value >= 0) && (value <= 1))    b->opt_zero_copy = value;
    else if (!strcmp(name, "eager") && (value >= 0) && (value <= 1))        b->opt_eager = value;
    else if (!strcmp(name, "early_pend") && (value >= 0) && (value <= 2))   b->opt_early_pend = value;
    else if (!strcmp(name, "early_src") && (value >= 0) && (value <= 2))    b->opt_early_src = value;
    else if (!strcmp(name, "lookahead") && ((value == -1) || (value == 0) || (value == 2) || (value == 4) || (value == 8)))
        b->opt_lookahead = value;
    else if (!strcmp(name, "multi_frame") && ((value == 0) || (value == 1) || (value == 2) || (value == 4) || (value == 8)))
        b->opt_multi = (value == 1) ? 0 : value;
    else
        return fail(B200CONV_ERR_ARG, "b200conv_set_option: unknown option or bad value: %s = %d", name, value);
    b->desc_dirty   = true;     /* the hand-shake counters are re-seeded before the next launch */
    b->pend_ready   = false;
    return B200CONV_OK;
}

extern "C" const char *b200conv_last_error(void)
{
    return g_last_error.c_str();
}

extern "C" const char *b200conv_version(void)
{
    return "b200conv 0.1 (sm_100a)";
}

/* ------------------------------------------------------------------------------------------- */
/* fused cross-GPU reduce (partition-range sharding)                                            */

extern "C" int b200conv_reduce_prepare(b200conv_batch_t *b, int grank, int world, unsigned char *handle_out)
{
    if ((b == nullptr) || (handle_out == nullptr) || (world < 1) || (world > REDUCE_MAX_WORLD) ||
        (grank < 0) || (grank >= world))
        return fail(B200CONV_ERR_ARG, "b200conv_reduce_prepare: bad arguments");
    if ((b->rank == 0) || (b->rank > 13))
        return fail(B200CONV_ERR_STATE, "b200conv_reduce_prepare: initialise the instances first (ranks 8..13)");
    static_assert(sizeof(cudaIpcMemHandle_t) == B200CONV_IPC_HANDLE_BYTES, "IPC handle size");
    ENTER_DEVICE(b);
    TRY(b200conv_reduce_disconnect(b));

    /* exchange buffer (identical layout on every rank):
     *   words    [DEPTH][world][channels][F] x { sample bits, sequence number = block + 1 }
     *   consumed [world][channels]           blocks consumed, written by the consuming rank
     *   scratch  [FRAME_SLOTS][channels][F]  this rank's own block, one per launch in flight (local) */
    const size_t F          = size_t(1) << (b->rank - 1);
    const size_t C          = b->n;
    b->xchg_slots_bytes     = size_t(REDUCE_DEPTH) * world * C * F * sizeof(uint2);
    b->xchg_consumed_off    = (b->xchg_slots_bytes + 127) & ~size_t(127);
    b->xchg_flags_off       = (b->xchg_consumed_off + size_t(world) * C * sizeof(uint32_t) + 127) & ~size_t(127);   /* scratch */
    size_t total            = b->xchg_flags_off + size_t(FRAME_SLOTS) * C * F * sizeof(float);
    CU(cudaMalloc(&b->xchg, total));
    CU(cudaMemset(b->xchg, 0, total));
    cudaIpcMemHandle_t hnd;
    CU(cudaIpcGetMemHandle(&hnd, b->xchg));
    memcpy(handle_out, &hnd, sizeof(hnd));

    memset(&b->reduce, 0, sizeof(b->reduce));
    b->reduce.world         = uint32_t(world);
    b->reduce.grank         = uint32_t(grank);
    b->reduce.channels      = uint32_t(C);
    b->reduce.frame         = uint32_t(F);
    return B200CONV_OK;
}

extern "C" int b200conv_reduce_connect(b200conv_batch_t *b, const unsigned char *all_handles)
{
    if ((b == nullptr) || (all_handles == nullptr) || (b->xchg == nullptr))
        return fail(B200CONV_ERR_ARG, "b200conv_reduce_connect: call b200conv_reduce_prepare first");
    ENTER_DEVICE(b);
    CU(quiesce(b));
    ReduceArgs &r = b->reduce;

    /* every active instance must sit at the same whole-frame count */
    uint64_t frames = 0;
    bool first = true;
    for (uint32_t i : b->active)
    {
        const Instance &in = b->inst[i];
        if ((in.off != 0) || ((!first) && (in.frames != frames)))
            return fail(B200CONV_ERR_STATE, "b200conv_reduce_connect: instances are not frame-aligned");
        frames  = in.frames;
        first   = false;
    }

    /* all-to-all: every rank opens every peer's exchange buffer */
    for (uint32_t g = 0; g < r.world; ++g)
    {
        b->xchg_peer[g] = nullptr;
        if (g == r.grank)
            continue;
        cudaIpcMemHandle_t hnd;
        memcpy(&hnd, all_handles + size_t(g) * B200CONV_IPC_HANDLE_BYTES, sizeof(hnd));
        CU(cudaIpcOpenMemHandle(&b->xchg_peer[g], hnd, cudaIpcMemLazyEnablePeerAccess));
    }
    for (uint32_t g = 0; g < r.world; ++g)
    {
        unsigned char *base = (g == r.grank) ? b->xchg : static_cast<unsigned char *>(b->xchg_peer[g]);
        r.words[g]          = reinterpret_cast<uint2 *>(base);
        r.consumed[g]       = reinterpret_cast<uint32_t *>(base + b->xchg_consumed_off);
    }
    r.scratch               = reinterpret_cast<float *>(b->xchg + b->xchg_flags_off);
    r.t0                    = uint32_t(frames);
    r.mode                  = (r.world > 1) ? 1u : 0u;
    *b->h_error             = 0;
    return B200CONV_OK;
}

extern "C" int b200conv_reduce_disconnect(b200conv_batch_t *b)
{
    if (b == nullptr)
        return fail(B200CONV_ERR_ARG, "b200conv_reduce_disconnect: NULL handle");
    if (b->xchg == nullptr)
        return B200CONV_OK;
    ENTER_DEVICE(b);
    if (b->stream)
        cudaStreamSynchronize(b->stream);
    cudaDeviceSynchronize();
    for (int g = 0; g < REDUCE_MAX_WORLD; ++g)
    {
        if (b->xchg_peer[g] != nullptr)
            cudaIpcCloseMemHandle(b->xchg_peer[g]);
        b->xchg_peer[g] = nullptr;
    }
    cudaFree(b->xchg);
    b->xchg = nullptr;
    memset(&b->reduce, 0, sizeof(b->reduce));
    return B200CONV_OK;
}

extern "C" int b200conv_reduce_status(b200conv_batch_t *b, int *timed_out)
{
    if ((b == nullptr) || (timed_out == nullptr))
        return fail(B200CONV_ERR_ARG, "b200conv_reduce_status: bad arguments");
    *timed_out = (b->h_error != nullptr) ? int(*reinterpret_cast<volatile uint32_t *>(b->h_error)) : 0;
    return B200CONV_OK;
}

/* ------------------------------------------------------------------------------------------- */
/* fastconv primitives on the device                                                            */

/* Stream-ordered: nothing here synchronises, takes a lock on the data path or uploads a job list.
 * Problem i lives at row i of each operand, so the kernels derive their jobs from the base
 * pointers (STEP_LINEAR_JOBS); scratch comes from the stream-ordered allocator
 * (cudaMallocAsync / cudaFreeAsync on the caller's stream).  The only shared state is the
 * per-device twiddle table of a rank, built once. */
namespace
{
    std::mutex  g_prim_lock;
    float2     *g_prim_tw[MAX_DEVICES][B200CONV_RANK_MAX + 1] = { { nullptr } };

    int prim_twiddles(int device, size_t rank, size_t count, float2 **tw)
    {
        if ((rank < B200CONV_RANK_MIN) || (rank > B200CONV_RANK_MAX) || (count == 0) || (count >= (size_t(1) << 31)))
            return fail(B200CONV_ERR_ARG, "fastconv: rank %zu / count %zu not supported", rank, count);
        int n = 0;
        cudaError_t e = cudaGetDeviceCount(&n);
        if ((e != cudaSuccess) || (n == 0))
            return fail(B200CONV_ERR_CUDA, "no CUDA device available (%s)", cudaGetErrorString(e));
        if ((device < 0) || (device >= n) || (device >= MAX_DEVICES))
            return fail(B200CONV_ERR_ARG, "device %d out of range", device);
        std::lock_guard<std::mutex> lock(g_prim_lock);      /* first use of a (device, rank) builds the table */
        if (g_prim_tw[device][rank] == nullptr)
            TRY(make_twiddles(uint32_t(rank), &g_prim_tw[device][rank]));
        *tw         = g_prim_tw[device][rank];
        return B200CONV_OK;
    }

    /* job i: transform input src + i * F, spectrum row spec + i * M, inverse output dst + i * dst_step */
    StepArgs prim_args(const float2 *tw, size_t rank, size_t count, const float *src, float *fwd_out_or_inv_dst,
                       size_t dst_step, uint32_t flags)
    {
        StepArgs a;
        memset(&a, 0, sizeof(a));
        a.tw        = tw;
        a.rank      = uint32_t(rank);
        a.n_jobs    = uint32_t(count);
        a.splits    = 1;
        a.src       = src;
        a.dst       = fwd_out_or_inv_dst;
        a.stride_dst = dst_step;
        a.flags     = STEP_LINEAR_JOBS | flags;
        return a;
    }

    /* ranks 13..16: scratch for the half-frame inverse (NULL when the launch will not use it) */
    int prim_park(size_t rank, size_t count, cudaStream_t st, float **park)
    {
        *park       = nullptr;
        if ((rank < 13) || ((rank < 16) && (count > 2 * MAX_FEW_JOBS)))
            return B200CONV_OK;
        CU(cudaMallocAsync(park, count * (size_t(2) << (rank - 1)) * sizeof(float), st));
        return B200CONV_OK;
    }
}

/* device < 0 = the calling thread's current device */
#define ENTER_PRIM_DEVICE(device)                                                           \
    if ((device) < 0)                                                                       \
        cudaGetDevice(&(device));                                                           \
    DeviceScope device_scope_(device);                                                      \
    if (device_scope_.error() != cudaSuccess)                                               \
        return fail(B200CONV_ERR_CUDA, "cannot select device %d: %s", (device),             \
                    cudaGetErrorString(device_scope_.error()))

extern "C" int b200conv_fastconv_parse(int device, float *image, const float *src, size_t rank,
                                       size_t count, void *stream)
{
    ENTER_PRIM_DEVICE(device);
    float2 *tw = nullptr;
    TRY(prim_twiddles(device, rank, count, &tw));
    if ((image == nullptr) || (src == nullptr))
        return fail(B200CONV_ERR_ARG, "b200conv_fastconv_parse: NULL buffer");
    StepArgs a = prim_args(tw, rank, count, src, image, 0, 0);
    CU(launch_fwd(a, uint32_t(count), cudaStream_t(stream)));
    return B200CONV_OK;
}

/* dst[i][0 .. 2^rank) (+)= IFFT(images[i]) / 2^rank; `images` may be clobbered by nobody: the
 * inverse reads it once */
static int prim_inverse(const float2 *tw, float *dst, const float2 *images, size_t rank, size_t count,
                        bool accumulate, cudaStream_t st)
{
    const size_t N  = size_t(1) << rank;
    float *rows = nullptr, *park = nullptr;
    if (accumulate)
        CU(cudaMallocAsync(&rows, count * N * sizeof(float), st));
    int rc = prim_park(rank, count, st, &park);
    if (rc == B200CONV_OK)
    {
        StepArgs a  = prim_args(tw, rank, count, nullptr, accumulate ? rows : dst, N, INV_FULL);
        a.ypart     = const_cast<float2 *>(images);
        a.park      = park;
        cudaError_t e = launch_inv(a, uint32_t(count), st);
        if ((e == cudaSuccess) && accumulate)
        {
            uint64_t total  = uint64_t(count) * N;
            uint32_t grid   = uint32_t((total + 255) / 256 > 4096 ? 4096 : (total + 255) / 256);
            k_accumulate<<<grid, 256, 0, st>>>(dst, rows, total);
            e               = cudaGetLastError();
        }
        if (e != cudaSuccess)
            rc              = fail(B200CONV_ERR_CUDA, "fastconv inverse failed: %s", cudaGetErrorString(e));
    }
    if (rows)   cudaFreeAsync(rows, st);
    if (park)   cudaFreeAsync(park, st);
    return rc;
}

extern "C" int b200conv_fastconv_restore(int device, float *dst, const float *image, size_t rank,
                                         size_t count, void *stream)
{
    ENTER_PRIM_DEVICE(device);
    float2 *tw = nullptr;
    TRY(prim_twiddles(device, rank, count, &tw));
    if ((dst == nullptr) || (image == nullptr))
        return fail(B200CONV_ERR_ARG, "b200conv_fastconv_restore: NULL buffer");
    return prim_inverse(tw, dst, reinterpret_cast<const float2 *>(image), rank, count, false, cudaStream_t(stream));
}

extern "C" int b200conv_fastconv_apply(int device, float *dst, const float *c1, const float *c2,
                                       size_t rank, size_t count, void *stream)
{
    ENTER_PRIM_DEVICE(device);
    float2 *tw = nullptr;
    TRY(prim_twiddles(device, rank, count, &tw));
    if ((dst == nullptr) || (c1 == nullptr) || (c2 == nullptr))
        return fail(B200CONV_ERR_ARG, "b200conv_fastconv_apply: NULL buffer");
    cudaStream_t st = cudaStream_t(stream);
    const size_t M  = size_t(1) << (rank - 1);
    float2 *prod    = nullptr;
    CU(cudaMallocAsync(&prod, count * M * sizeof(float2), st));
    uint64_t total  = uint64_t(count) * M;
    uint32_t grid   = uint32_t((total + 255) / 256 > 4096 ? 4096 : (total + 255) / 256);
    k_cmul<<<grid, 256, 0, st>>>(prod, reinterpret_cast<const float2 *>(c1),
                                 reinterpret_cast<const float2 *>(c2), uint32_t(M), total);
    int rc = (cudaGetLastError() == cudaSuccess) ? prim_inverse(tw, dst, prod, rank, count, true, st)
                                                 : fail(B200CONV_ERR_CUDA, "k_cmul launch failed");
    cudaFreeAsync(prod, st);
    return rc;
}

extern "C" int b200conv_fastconv_parse_apply(int device, float *dst, const float *cimg, const float *src,
                                             size_t rank, size_t count, void *stream)
{
    ENTER_PRIM_DEVICE(device);
    float2 *tw = nullptr;
    TRY(prim_twiddles(device, rank, count, &tw));
    if ((dst == nullptr) || (cimg == nullptr) || (src == nullptr))
        return fail(B200CONV_ERR_ARG, "b200conv_fastconv_parse_apply: NULL buffer");
    cudaStream_t st = cudaStream_t(stream);
    const size_t M  = size_t(1) << (rank - 1);
    float2 *prod    = nullptr;
    CU(cudaMallocAsync(&prod, count * M * sizeof(float2), st));
    StepArgs a      = prim_args(tw, rank, count, src, reinterpret_cast<float *>(prod), 0, 0);
    cudaError_t e   = launch_fwd(a, uint32_t(count), st);
    if (e == cudaSuccess)
    {
        uint64_t total  = uint64_t(count) * M;
        uint32_t grid   = uint32_t((total + 255) / 256 > 4096 ? 4096 : (total + 255) / 256);
        k_cmul<<<grid, 256, 0, st>>>(prod, prod, reinterpret_cast<const float2 *>(cimg), uint32_t(M), total);
        e               = cudaGetLastError();
    }
    int rc = (e == cudaSuccess) ? prim_inverse(tw, dst, prod, rank, count, true, st)
                                : fail(B200CONV_ERR_CUDA, "fastconv_parse_apply failed: %s", cudaGetErrorString(e));
    cudaFreeAsync(prod, st);
    return rc;
}

extern "C" int b200conv_convolve(int device, float *dst, size_t dst_stride, const float *src, size_t src_stride,
                                 const float *conv, size_t conv_stride, size_t length, size_t count,
                                 size_t batch, void *stream)
{
    if ((dst == nullptr) || (src == nullptr) || (conv == nullptr) || (batch > 65535) ||
        (length >= (size_t(1) << 31)) || (count >= (size_t(1) << 31)))
        return fail(B200CONV_ERR_ARG, "b200conv_convolve: bad arguments");
    if ((length == 0) || (count == 0) || (batch == 0))
        return B200CONV_OK;
    ENTER_PRIM_DEVICE(device);
    size_t n        = count + length - 1;
    dim3 grid(uint32_t((n + 127) / 128 > 1024 ? 1024 : (n + 127) / 128), uint32_t(batch));
    k_convolve<<<grid, 128, 0, cudaStream_t(stream)>>>(dst, dst_stride, src, src_stride, conv, conv_stride,
                                                       uint32_t(length), uint32_t(count));
    CU(cudaGetLastError());
    return B200CONV_OK;
}

/* ------------------------------------------------------------------------------------------- */
/* offline linear convolution                                                                   */

extern "C" int b200conv_linear_convolve(int device, float *dst, size_t dst_stride, const float *src,
                                        size_t src_stride, size_t nx, size_t count, const float *h,
                                        size_t nh, size_t rank)
{
    if ((dst == nullptr) || (src == nullptr) || (h == nullptr) || (nx == 0) || (nh == 0) || (count == 0) ||
        (src_stride < nx) || (dst_stride < nx + nh - 1))
        return fail(B200CONV_ERR_ARG, "b200conv_linear_convolve: bad arguments");

    b200conv_batch_t *b = nullptr;
    TRY(b200conv_create(&b, device, count));
    int rc = B200CONV_OK;
    rc = b200conv_init(b, 0, h, nh, rank, 0.0f);                /* ONE set of filter spectra ... */
    for (size_t i = 1; (i < count) && (rc == B200CONV_OK); ++i)
        rc = b200conv_init_shared(b, i, 0, 0.0f);               /* ... borrowed by every other signal */

    float *in = nullptr, *out = nullptr;
    if (rc == B200CONV_OK)
    {
        const size_t F      = size_t(1) << (b->rank - 1);
        const size_t total  = ((nx + nh - 1 + F - 1) / F) * F;     /* whole frames: the fast path */
        if ((cudaMallocHost(&in, count * total * sizeof(float)) != cudaSuccess) ||
            (cudaMallocHost(&out, count * total * sizeof(float)) != cudaSuccess))
            rc = fail(B200CONV_ERR_NOMEM, "b200conv_linear_convolve: out of page-locked host memory");
        else
        {
            memset(in, 0, count * total * sizeof(float));
            for (size_t i = 0; i < count; ++i)
                memcpy(in + i * total, src + i * src_stride, nx * sizeof(float));
            rc = b200conv_process_planar(b, out, in, total, total);
            if (rc == B200CONV_OK)
                for (size_t i = 0; i < count; ++i)
                    memcpy(dst + i * dst_stride, out + i * total, (nx + nh - 1) * sizeof(float));
        }
    }
    std::string keep = g_last_error;
    if (in)  cudaFreeHost(in);
    if (out) cudaFreeHost(out);
    b200conv_free(b);
    g_last_error = keep;
    return rc;
}

/* ------------------------------------------------------------------------------------------- */
/* SyncChirpProcessor::do_linear_convolutions                                                   */

static const size_t CHIRP_MAX_PART_SIZE = 32768;            /* MAX_PART_SIZE, SyncChirpProcessor.cpp:43 */

extern "C" int b200conv_chirp_plan(b200conv_chirp_plan_t *plan, size_t *partitions, size_t *padded,
                                   size_t *prepends, size_t *conv_lengths, size_t *align_offsets,
                                   const size_t *in_len, size_t nchannels, size_t inverse_len,
                                   size_t part_size_limit)
{
    if ((plan == nullptr) || (in_len == nullptr) || (nchannels == 0))
        return fail(B200CONV_ERR_ARG, "b200conv_chirp_plan: bad arguments");       /* STATUS_NO_DATA, :1376 */
    /* the partition: a power of two, at most MAX_PART_SIZE, 0 = MAX_PART_SIZE (:1226-1240) */
    size_t limit        = (part_size_limit < CHIRP_MAX_PART_SIZE) ? part_size_limit : CHIRP_MAX_PART_SIZE;
    if (limit == 0)
        limit               = CHIRP_MAX_PART_SIZE;
    size_t log2p        = 0;
    while ((size_t(1) << log2p) < limit)
        ++log2p;
    const size_t P      = size_t(1) << log2p;
    plan->partition_size    = P;
    plan->conv_rank         = log2p + 1;
    plan->image             = size_t(1) << (log2p + 2);
    plan->allocation_size   = 0;
    /* both sequences are thought of as padded to a whole number of partitions, the recording at
     * its tail, the inverse filter at its head (:1313-1323) */
    for (size_t ch = 0; ch < nchannels; ++ch)
    {
        const size_t longest    = (in_len[ch] > inverse_len) ? in_len[ch] : inverse_len;
        const size_t np         = longest / P + 1;
        if (partitions)     partitions[ch]      = np;
        if (padded)         padded[ch]          = np * P;
        if (prepends)       prepends[ch]        = np * P - inverse_len;
        if (conv_lengths)   conv_lengths[ch]    = 2 * np * P;
        if (2 * np * P > plan->allocation_size)
            plan->allocation_size   = 2 * np * P;
    }
    /* rows are centred on the middle of the longest one (:1327-1330) */
    if (align_offsets)
        for (size_t ch = 0; ch < nchannels; ++ch)
        {
            const size_t longest    = (in_len[ch] > inverse_len) ? in_len[ch] : inverse_len;
            align_offsets[ch]       = plan->allocation_size / 2 - (longest / P + 1) * P;
        }
    return B200CONV_OK;
}

static int chirp_impl(int device, float *result, size_t result_stride, const float *const *inputs,
                      const size_t *in_len, size_t nchannels, const float *inverse, size_t inverse_len,
                      size_t part_size_limit, float scale)
{
    if ((result == nullptr) || (inputs == nullptr) || (in_len == nullptr) || (nchannels == 0) ||
        (inverse == nullptr) || (inverse_len == 0))
        return fail(B200CONV_ERR_ARG, "b200conv_chirp_linear_convolutions: bad arguments");
    for (size_t ch = 0; ch < nchannels; ++ch)
        if ((inputs[ch] == nullptr) && (in_len[ch] > 0))
            return fail(B200CONV_ERR_ARG, "b200conv_chirp_linear_convolutions: NULL input for channel %zu", ch);

    std::vector<size_t> parts(nchannels), padded(nchannels), prepends(nchannels), clen(nchannels), align(nchannels);
    b200conv_chirp_plan_t plan;
    TRY(b200conv_chirp_plan(&plan, parts.data(), padded.data(), prepends.data(), clen.data(), align.data(),
                            in_len, nchannels, inverse_len, part_size_limit));
    if ((plan.conv_rank < B200CONV_RANK_MIN) || (plan.conv_rank > B200CONV_RANK_MAX))
        return fail(B200CONV_ERR_ARG, "partition size %zu (rank %zu) is outside the engine's ranks 8..16",
                    plan.partition_size, plan.conv_rank);
    if (result_stride < plan.allocation_size)
        return fail(B200CONV_ERR_ARG, "result rows must hold %zu samples", plan.allocation_size);

    const size_t P      = plan.partition_size;
    size_t frames       = 0;                            /* every channel: 2 * vPartitions frames of P samples */
    for (size_t ch = 0; ch < nchannels; ++ch)
        frames              = (2 * parts[ch] > frames) ? 2 * parts[ch] : frames;
    const size_t total  = frames * P;

    b200conv_batch_t *b = nullptr;
    TRY(b200conv_create(&b, device, nchannels));
    int rc = B200CONV_OK;
    {
        /* the prepend-padded inverse filter is the impulse response; channels of equal padded
         * length see the same one and share its spectra */
        std::vector<float> ir;
        for (size_t ch = 0; (ch < nchannels) && (rc == B200CONV_OK); ++ch)
        {
            size_t same         = ch;
            for (size_t k = 0; k < ch; ++k)
                if (padded[k] == padded[ch]) { same = k; break; }
            if (same != ch)
            {
                rc                  = b200conv_init_shared(b, ch, same, 0.0f);
                continue;
            }
            ir.assign(padded[ch], 0.0f);
            memcpy(ir.data() + prepends[ch], inverse, inverse_len * sizeof(float));
            rc                  = b200conv_init(b, ch, ir.data(), ir.size(), plan.conv_rank, 0.0f);
        }
    }
    if (rc == B200CONV_OK)
    {
        std::vector<float> in(nchannels * total, 0.0f), out(nchannels * total);
        for (size_t ch = 0; ch < nchannels; ++ch)
            if (in_len[ch] > 0)
                memcpy(in.data() + ch * total, inputs[ch], in_len[ch] * sizeof(float));
        rc = b200conv_process_planar(b, out.data(), in.data(), total, total);
        if (rc == B200CONV_OK)
            for (size_t ch = 0; ch < nchannels; ++ch)
            {
                float *row          = result + ch * result_stride;
                memset(row, 0, plan.allocation_size * sizeof(float));       /* allocateConvolutionResult */
                memcpy(row + align[ch], out.data() + ch * total, clen[ch] * sizeof(float));
                for (size_t i = 0; i < clen[ch]; ++i)                      /* :1508, from index 0 */
                    row[i]             *= scale;
            }
    }
    std::string keep = g_last_error;
    b200conv_free(b);
    g_last_error = keep;
    return rc;
}

extern "C" int b200conv_chirp_linear_convolutions(int device, float *result, size_t result_stride,
                                                  const float *const *inputs, const size_t *in_len,
                                                  size_t nchannels, const float *inverse, size_t inverse_len,
                                                  size_t part_size_limit, float scale)
{
    try { return chirp_impl(device, result, result_stride, inputs, in_len, nchannels, inverse, inverse_len,
                            part_size_limit, scale); }
    catch (const std::bad_alloc &) { return fail(B200CONV_ERR_NOMEM, "out of host memory"); }
}

#include "equalizer.cuh"
#include "spectral.cuh"
#include "spectral_host.cuh"
#include "splitter.cuh"
#include "matrix.cuh"
#include "matrix_host.cuh"

#ifdef B200CONV_TIMING
/* developer instrumentation: copies the per-CTA timestamps of the last k_frame launch */
extern "C" int b200conv_debug_frame_times(unsigned long long *out, size_t count)
{
    CU(cudaDeviceSynchronize());
    CU(cudaMemcpyFromSymbol(out, g_frame_times, count * sizeof(unsigned long long)));
    return B200CONV_OK;
}
#endif

/* ------------------------------------------------------------------------------------------- */
/* exception guards for the entry points that allocate host containers                          */

extern "C" int b200conv_create(b200conv_batch_t **out, int device, size_t instances)
{
    try { return create_impl(out, device, instances); }
    catch (const std::bad_alloc &) { return fail(B200CONV_ERR_NOMEM, "out of host memory"); }
}

extern "C" int b200conv_init_range(b200conv_batch_t *b, size_t idx, const float *data, size_t count,
                                   size_t rank, float phase, size_t part_offset)
{
    try { return init_range_impl(b, idx, data, count, rank, phase, part_offset); }
    catch (const std::bad_alloc &) { return fail(B200CONV_ERR_NOMEM, "out of host memory"); }
}

extern "C" int b200conv_init_shared(b200conv_batch_t *b, size_t idx, size_t src_idx, float phase)
{
    try { return init_shared_impl(b, idx, src_idx, phase); }
    catch (const std::bad_alloc &) { return fail(B200CONV_ERR_NOMEM, "out of host memory"); }
}

extern "C" int b200conv_init_many(b200conv_batch_t *b, size_t count, const size_t *idx, const float *const *data,
                                  const size_t *counts, size_t rank, const float *phases, const size_t *part_offsets)
{
    try { return init_many_impl(b, count, idx, data, counts, rank, phases, part_offsets); }
    catch (const std::bad_alloc &) { return fail(B200CONV_ERR_NOMEM, "out of host memory"); }
}

extern "C" int b200conv_process_device2(b200conv_batch_t *b, float *dst, size_t dst_stride,
                                        const float *src, size_t src_stride, size_t count, void *stream)
{
    try { return process_device2_impl(b, dst, dst_stride, src, src_stride, count, stream); }
    catch (const std::bad_alloc &) { return fail(B200CONV_ERR_NOMEM, "out of host memory"); }
}


/*
 * matrix_host.cuh -- host side and C ABI (b200conv_mx_*) of the matrix convolver (included by
 * engine.cu after matrix.cuh).
 *
 * Per launch group of up to MX_GROUP_FRAMES whole frames, three launches on one stream:
 *   k_fwd      one job per (frame, input): the caller's block -> the input's ring slot (-t) mod S;
 *              launched WITHOUT programmatic serialisation: it starts after everything before it has
 *              completed, in particular the k_inv of the previous group (the last reader of ypart);
 *   k_mx_mac   programmatic serialisation: it may start once every CTA of that k_fwd has started;
 *              it reads the new frame's ring row only after griddepcontrol.wait (matrix.cuh);
 *   k_inv      programmatic serialisation: one job per (frame, output) summing `rows` partial rows.
 * So when k_mx_mac(t) starts, k_fwd(t) has started, which it did only after k_inv(t - 1) completed:
 * the older ring rows and the partial rows it touches early are final.
 *
 * While a crossfade of b200conv_mx_set_irs runs, a group has one more launch: k_mx_blend, plain
 * stream order behind that k_inv, adds w * (delta outputs) into the outputs.  The group's k_mx_mac
 * reads a units table with the delta units appended and writes a ypart of its own.
 */
#ifndef B200CONV_MATRIX_HOST_CUH_
#define B200CONV_MATRIX_HOST_CUH_

#include <map>

static const size_t   MX_MAX_IO         = 4096;                 /* inputs, outputs per object */
static const uint32_t MX_GROUP_FRAMES   = 32;                   /* frames per launch group (bounds the ring's spare slots) */
static const size_t   MX_GROUP_JOBS     = size_t(1) << 13;      /* transform jobs per launch group */
static const size_t   MX_SCRATCH_BYTES  = size_t(256) << 20;    /* partial rows + half-frame scratch of one launch group */

struct MxRoute                              /* host mirror of one route */
{
    uint32_t        input, output, nq;      /* nq: rows of G */
    uint32_t        unit, slot;             /* where the units table holds it */
    const float2   *G;
    void           *owner;                  /* the stream-ordered allocation G lies in */
};

/* A crossfade in progress (b200conv_mx_set_irs).  Everything here is stream-ordered memory: it is
 * released on the stream of the call in which the fade ends. */
struct MxFade
{
    bool        active      = false;
    uint64_t    t0          = 0;            /* frame index of the fade's first sample */
    uint64_t    fade        = 0;            /* samples */
    MxUnit     *units       = nullptr;      /* the plan's units, then the delta units */
    MxUnit     *units_final = nullptr;      /* the plan's units with the new G: in use once the fade ends */
    float2     *ypart       = nullptr;      /* [zmax][outputs + deltas][rows][M] */
    float      *park        = nullptr;      /* ranks 13..16 */
    uint32_t   *tickets     = nullptr;
    float      *dout        = nullptr;      /* [zmax][deltas][F]: the delta outputs' blocks */
    uint32_t   *omap        = nullptr;      /* [deltas]: output of each delta output */
    float2     *D           = nullptr;      /* G_new - G_old of every changed route */
    uint32_t    n_units     = 0, rg = 1, zmax = 1, deltas = 0;
    size_t      smem        = 0;
    std::vector<size_t>         changed;    /* routes */
    std::vector<uint32_t>       nq_new;
    std::vector<float2 *>       G_new;      /* one allocation per changed route */
    std::vector<MxUnit>         host_final;
};

/* What one set_routes builds; swapped in whole, so that a failed call leaves the previous one intact. */
struct MxPlan
{
    size_t      routes      = 0;
    float2     *G           = nullptr;      /* every route's folded IR spectra, route after route */
    float2     *ring        = nullptr;      /* [inputs][S][M] */
    float2     *ypart       = nullptr;      /* [zmax][outputs][rows][M]; rows no route writes stay zero */
    float      *park        = nullptr;      /* ranks 13..16: k_inv_half scratch, [zmax * outputs][2][F] */
    uint32_t   *tickets     = nullptr;      /* ... and its per-job counters (zero between launches) */
    MxUnit     *units       = nullptr;
    uint32_t    n_units     = 0, rg = 1, splits = 1, rows = 1, zmax = 1, S = 0;
    uint32_t    nq_cap      = 0;            /* longest route's rows: the ring's reach for b200conv_mx_set_irs */
    size_t      ring_bytes  = 0;
    size_t      smem        = 0;
    std::vector<MxRoute>        rt;
    std::vector<MxUnit>         host_units; /* what `units` holds */
    std::map<void *, uint32_t>  owners;     /* G allocations and the routes that point into each */
    MxFade      fade;
};

struct b200conv_mx
{
    int         device      = 0;
    int         sm_count    = 148;
    size_t      I = 0, O = 0, rank = 0, F = 0;
    cudaStream_t stream     = nullptr;
    cudaEvent_t ev_last     = nullptr;      /* end of the latest call on a CALLER's stream */
    bool        last_foreign = false;
    float2     *tw          = nullptr;
    MxPlan      plan;
    uint64_t    t           = 0;            /* frames since set_routes / clear */

    /* job upload ring (page-locked), used in two halves (mx_reserve_jobs) */
    Job        *h_jobs      = nullptr;
    Job        *d_jobs      = nullptr;
    size_t      job_cap     = 0, job_pos = 0, job_half = 0;     /* job_pos lies in half job_half */
    cudaEvent_t ev_half[2]  = { nullptr, nullptr };
    bool        half_used[2] = { false, false };

    float      *sd_in = nullptr, *sd_out = nullptr;     /* process_planar staging */
    size_t      stage_cols  = 0;

    unsigned char *h_irs    = nullptr;      /* set_irs staging (page-locked) */
    size_t      irs_cap     = 0;
    cudaEvent_t ev_irs      = nullptr;      /* the uploads that last read h_irs */
    bool        irs_used    = false;
};

typedef b200conv_mx Mx;

static void mx_free_async(void *ptr, cudaStream_t st)
{
    if (ptr)
        cudaFreeAsync(ptr, st);
}

/* the fade's buffers; its new G only when `with_g` (otherwise they now belong to routes) */
static void mx_fade_free(MxFade &f, bool with_g, cudaStream_t st)
{
    mx_free_async(f.units, st);
    mx_free_async(f.ypart, st);
    mx_free_async(f.park, st);
    mx_free_async(f.tickets, st);
    mx_free_async(f.dout, st);
    mx_free_async(f.omap, st);
    mx_free_async(f.D, st);
    if (with_g)
    {
        mx_free_async(f.units_final, st);
        for (float2 *g : f.G_new)
            mx_free_async(g, st);
    }
    f = MxFade();
}

/* G and the units tables are stream-ordered allocations (b200conv_mx_set_irs releases them while
 * the device runs); the ring and the scratch of set_routes are not */
static void mx_plan_free(MxPlan &p, cudaStream_t st)
{
    mx_fade_free(p.fade, true, st);
    for (const auto &o : p.owners)
        mx_free_async(o.first, st);
    mx_free_async(p.units, st);
    if (p.ring)     cudaFree(p.ring);
    if (p.ypart)    cudaFree(p.ypart);
    if (p.park)     cudaFree(p.park);
    if (p.tickets)  cudaFree(p.tickets);
    p = MxPlan();
}

/* The fade is over: the changed routes take their new G for good, the units table without the
 * delta units takes over, and what only the fade (or the old IRs) needed is released on `st`,
 * behind every launch that reads it. */
static int mx_fade_finish(Mx *m, cudaStream_t st)
{
    MxPlan &p   = m->plan;
    MxFade &f   = p.fade;
    if (!f.active)
        return B200CONV_OK;
    for (size_t k = 0; k < f.changed.size(); ++k)
    {
        MxRoute &r      = p.rt[f.changed[k]];
        auto it         = p.owners.find(r.owner);
        if ((it != p.owners.end()) && (--it->second == 0))
        {
            mx_free_async(it->first, st);
            p.owners.erase(it);
        }
        r.G             = f.G_new[k];
        r.nq            = f.nq_new[k];
        r.owner         = f.G_new[k];
        p.owners[r.owner] = 1;
    }
    mx_free_async(p.units, st);
    p.units         = f.units_final;
    p.host_units    = f.host_final;
    mx_fade_free(f, false, st);
    CU(cudaGetLastError());
    return B200CONV_OK;
}

/* everything enqueued on the object, on its own stream and on a caller's */
static cudaError_t mx_quiesce(Mx *m)
{
    cudaError_t e = cudaStreamSynchronize(m->stream);
    if ((e == cudaSuccess) && m->last_foreign)
        e = cudaEventSynchronize(m->ev_last);
    m->last_foreign = false;
    return e;
}

extern "C" void b200conv_mx_free(b200conv_mx_t *m)
{
    if (m == nullptr)
        return;
    DeviceScope device_scope_(m->device);
    if (m->stream)
    {
        mx_quiesce(m);
        mx_plan_free(m->plan, m->stream);
        cudaStreamSynchronize(m->stream);
    }
    if (m->tw)      cudaFree(m->tw);
    if (m->h_irs)   cudaFreeHost(m->h_irs);
    if (m->ev_irs)  cudaEventDestroy(m->ev_irs);
    if (m->h_jobs)  cudaFreeHost(m->h_jobs);
    if (m->d_jobs)  cudaFree(m->d_jobs);
    if (m->sd_in)   cudaFree(m->sd_in);
    if (m->sd_out)  cudaFree(m->sd_out);
    for (cudaEvent_t ev : m->ev_half)
        if (ev)     cudaEventDestroy(ev);
    if (m->ev_last) cudaEventDestroy(m->ev_last);
    if (m->stream)  cudaStreamDestroy(m->stream);
    delete m;
}

static int mx_create_impl(b200conv_mx_t **out, int device, size_t inputs, size_t outputs, size_t rank)
{
    if ((out == nullptr) || (inputs == 0) || (outputs == 0) || (inputs > MX_MAX_IO) || (outputs > MX_MAX_IO) ||
        (rank < B200CONV_RANK_MIN) || (rank > B200CONV_RANK_MAX))
        return fail(B200CONV_ERR_ARG, "b200conv_mx_create: bad arguments (1..%zu inputs and outputs, ranks %d..%d)",
                    MX_MAX_IO, B200CONV_RANK_MIN, B200CONV_RANK_MAX);
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if ((e != cudaSuccess) || (count == 0))
        return fail(B200CONV_ERR_CUDA, "no CUDA device available (%s); this engine has no CPU fallback", cudaGetErrorString(e));
    if (device < 0)
        CU(cudaGetDevice(&device));
    if (device >= count)
        return fail(B200CONV_ERR_ARG, "device %d out of range (%d devices)", device, count);

    Mx *m = new (std::nothrow) Mx();
    if (m == nullptr)
        return fail(B200CONV_ERR_NOMEM, "out of host memory");
    m->device   = device;
    m->I        = inputs;
    m->O        = outputs;
    m->rank     = rank;
    m->F        = size_t(1) << (rank - 1);
    /* two halves, each holding the jobs of the largest launch group: MX_GROUP_JOBS, or one frame of a
     * fade (I inputs, O outputs and up to O delta outputs) when that is more */
    m->job_cap  = 2 * std::max(MX_GROUP_JOBS, inputs + 2 * outputs);

    ENTER_DEVICE(m);
    int rc = B200CONV_OK;
    do
    {
        cudaDeviceProp prop;
        if (cudaGetDeviceProperties(&prop, device) == cudaSuccess)
            m->sm_count = prop.multiProcessorCount;
        #define CU_BRK(call) { cudaError_t e_ = (call); if (e_ != cudaSuccess) { rc = fail((e_ == cudaErrorMemoryAllocation) ? B200CONV_ERR_NOMEM : B200CONV_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(e_)); break; } }
        CU_BRK(cudaStreamCreateWithFlags(&m->stream, cudaStreamNonBlocking));
        CU_BRK(cudaEventCreateWithFlags(&m->ev_last, cudaEventDisableTiming));
        CU_BRK(cudaEventCreateWithFlags(&m->ev_half[0], cudaEventDisableTiming));
        CU_BRK(cudaEventCreateWithFlags(&m->ev_half[1], cudaEventDisableTiming));
        CU_BRK(cudaEventCreateWithFlags(&m->ev_irs, cudaEventDisableTiming));
        CU_BRK(cudaMallocHost(&m->h_jobs, m->job_cap * sizeof(Job)));
        CU_BRK(cudaMalloc(&m->d_jobs, m->job_cap * sizeof(Job)));
        #undef CU_BRK
        if (rc == B200CONV_OK)
            rc = make_twiddles(uint32_t(rank), &m->tw);
    } while (false);
    if (rc != B200CONV_OK)
    {
        std::string keep = g_last_error;
        b200conv_mx_free(m);
        g_last_error = keep;
        return rc;
    }
    *out = m;
    return B200CONV_OK;
}

extern "C" int b200conv_mx_create(b200conv_mx_t **out, int device, size_t inputs, size_t outputs, size_t rank)
{
    try { return mx_create_impl(out, device, inputs, outputs, rank); }
    catch (const std::bad_alloc &) { return fail(B200CONV_ERR_NOMEM, "out of host memory"); }
}

static int mx_set_routes_impl(b200conv_mx_t *m, size_t count, const size_t *input, const size_t *output,
                              const float *const *ir, const size_t *length)
{
    if (m == nullptr)
        return fail(B200CONV_ERR_ARG, "b200conv_mx_set_routes: NULL handle");
    if ((count > 0) && ((input == nullptr) || (output == nullptr) || (ir == nullptr) || (length == nullptr)))
        return fail(B200CONV_ERR_ARG, "b200conv_mx_set_routes: NULL array");
    if (count > m->I * m->O)
        return fail(B200CONV_ERR_ARG, "b200conv_mx_set_routes: %zu routes, at most one per (input, output) pair", count);
    const size_t F = m->F, M = F, rank = m->rank;

    std::vector<uint64_t> pairs(count);
    size_t rows_total = 0, nq_max = 0, g_rows = 0;
    for (size_t r = 0; r < count; ++r)
    {
        if ((input[r] >= m->I) || (output[r] >= m->O))
            return fail(B200CONV_ERR_ARG, "route %zu: input %zu / output %zu out of range", r, input[r], output[r]);
        if ((ir[r] == nullptr) || (length[r] == 0))
            return fail(B200CONV_ERR_ARG, "route %zu: NULL or empty impulse response", r);
        const size_t bins = (length[r] >> (rank - 1)) + (((length[r] & (F - 1)) != 0) ? 1 : 0);    /* no wrap */
        if (bins + 1 >= (size_t(1) << 30))
            return fail(B200CONV_ERR_ARG, "route %zu: impulse response too long", r);
        pairs[r]        = uint64_t(input[r]) * m->O + output[r];
        rows_total     += bins;
        g_rows         += bins + 1;
        nq_max          = (bins + 1 > nq_max) ? bins + 1 : nq_max;
    }
    {
        std::vector<uint64_t> sorted(pairs);
        std::sort(sorted.begin(), sorted.end());
        if (std::adjacent_find(sorted.begin(), sorted.end()) != sorted.end())
            return fail(B200CONV_ERR_ARG, "b200conv_mx_set_routes: an (input, output) pair appears twice");
    }

    ENTER_DEVICE(m);
    CU(mx_quiesce(m));              /* ordered after every call already enqueued */
    cudaStream_t st = m->stream;

    /* ---- the plan: groups of up to MX_RG routes per input, rank among the routes into each output */
    MxPlan p;
    p.routes        = count;
    std::vector<uint32_t> fan_in(m->O, 0), rank_in(count, 0);
    uint32_t fan_max = 0;
    for (size_t r = 0; r < count; ++r)
    {
        rank_in[r]      = fan_in[output[r]]++;
        fan_max         = (fan_in[output[r]] > fan_max) ? fan_in[output[r]] : fan_max;
    }
    std::vector<std::vector<size_t>> leaving(m->I);
    for (size_t r = 0; r < count; ++r)
        leaving[input[r]].push_back(r);
    std::vector<MxUnit> units;
    std::vector<size_t> g_off(count, 0);
    for (size_t r = 1; r < count; ++r)
        g_off[r]        = g_off[r - 1] + ((length[r - 1] + F - 1) >> (rank - 1)) + 1;
    for (size_t i = 0; i < m->I; ++i)
        for (size_t k0 = 0; k0 < leaving[i].size(); k0 += MX_RG)
        {
            MxUnit u;
            memset(&u, 0, sizeof(u));
            u.input         = uint32_t(i);
            u.nr            = uint32_t(std::min<size_t>(MX_RG, leaving[i].size() - k0));
            p.rg            = (u.nr > p.rg) ? u.nr : p.rg;
            units.push_back(u);
        }
    p.n_units       = uint32_t(units.size());

    const uint32_t TB = uint32_t((M < 1024) ? M : 1024), QB = 1024 / TB, tiles = uint32_t(M / TB);
    p.smem          = size_t(MX_STAGES) * (1 + p.rg) * QB * TB * sizeof(float2) + MX_STAGES * sizeof(uint64_t) + 16;
    if (count > 0)
    {
        /* enough splits of the partition range for every SM to hold as many CTAs as fit (2 by the
         * launch bounds), at least two stages of work per split */
        size_t per_sm   = (227u * 1024u) / (p.smem + 1024u);
        per_sm          = (per_sm > 2) ? 2 : ((per_sm < 1) ? 1 : per_sm);
        const size_t ctas = size_t(p.n_units) * tiles;
        size_t splits   = (per_sm * size_t(m->sm_count)) / ctas;
        const size_t cap = nq_max / (2 * QB);
        splits          = (splits > cap) ? cap : splits;
        splits          = (splits > 32) ? 32 : ((splits < 1) ? 1 : splits);
        p.splits        = uint32_t(splits);
    }
    p.rows          = (fan_max > 0) ? fan_max * p.splits : 1;
    const size_t per_frame = m->O * p.rows * M * sizeof(float2) + ((rank >= 13) ? m->O * 2 * F * sizeof(float) : 0);
    size_t zmax     = MX_SCRATCH_BYTES / per_frame;
    zmax            = (zmax > MX_GROUP_FRAMES) ? MX_GROUP_FRAMES : zmax;
    zmax            = (zmax > MX_GROUP_JOBS / (m->I + m->O)) ? MX_GROUP_JOBS / (m->I + m->O) : zmax;
    p.zmax          = uint32_t((zmax < 1) ? 1 : zmax);
    p.S             = uint32_t(nq_max + p.zmax);    /* a group's newest frame never overwrites a row its oldest reads */
    p.ring_bytes    = m->I * size_t(p.S) * M * sizeof(float2);

    {
        size_t u_at = 0;
        for (size_t i = 0; i < m->I; ++i)
            for (size_t k0 = 0; k0 < leaving[i].size(); k0 += MX_RG, ++u_at)
            {
                MxUnit &u       = units[u_at];
                for (uint32_t k = 0; k < u.nr; ++k)
                {
                    const size_t r  = leaving[i][k0 + k];
                    const uint32_t nq = uint32_t(((length[r] + F - 1) >> (rank - 1)) + 1);
                    u.nq[k]         = nq;
                    u.row[k]        = uint32_t(output[r]) * p.rows + rank_in[r] * p.splits;
                    u.nq_max        = (nq > u.nq_max) ? nq : u.nq_max;
                }
            }
    }

    /* ---- allocate everything new before touching the old state */
    float *irdev = nullptr;
    float2 *H = nullptr;
    FoldDesc *d_fold = nullptr;
    cudaError_t e = cudaSuccess;
    auto alloc = [&](void **ptr, size_t bytes) { if ((e == cudaSuccess) && (bytes > 0)) e = cudaMalloc(ptr, bytes); };
    alloc(reinterpret_cast<void **>(&p.ring), p.ring_bytes);
    alloc(reinterpret_cast<void **>(&p.ypart), p.zmax * m->O * size_t(p.rows) * M * sizeof(float2));
    if (count > 0)
    {
        if (e == cudaSuccess)
            e = cudaMallocAsync(reinterpret_cast<void **>(&p.G), g_rows * M * sizeof(float2), st);
        if (e == cudaSuccess)
        {
            p.owners[p.G] = uint32_t(count);
            e = cudaMallocAsync(reinterpret_cast<void **>(&p.units), units.size() * sizeof(MxUnit), st);
        }
        alloc(reinterpret_cast<void **>(&irdev), rows_total * F * sizeof(float));
        alloc(reinterpret_cast<void **>(&H), rows_total * M * sizeof(float2));
        alloc(reinterpret_cast<void **>(&d_fold), count * sizeof(FoldDesc));
    }
    if (rank >= 13)
    {
        alloc(reinterpret_cast<void **>(&p.park), p.zmax * m->O * 2 * F * sizeof(float));
        alloc(reinterpret_cast<void **>(&p.tickets), p.zmax * m->O * sizeof(uint32_t));
    }
    auto drop_scratch = [&]()
    {
        if (irdev)  cudaFree(irdev);
        if (H)      cudaFree(H);
        if (d_fold) cudaFree(d_fold);
    };
    if (e != cudaSuccess)
    {
        cudaGetLastError();
        drop_scratch();
        mx_plan_free(p, st);
        return fail(B200CONV_ERR_NOMEM, "b200conv_mx_set_routes: allocation failed: %s", cudaGetErrorString(e));
    }

    /* ---- IR ingest: every partition of every route in one k_fwd launch, then one k_fold_many
     * (the b200conv_init_many path; calls are whole frames, so no time-domain head is kept) */
    int rc = B200CONV_OK;
    do
    {
        #define CU_BRK(call) { cudaError_t e_ = (call); if (e_ != cudaSuccess) { rc = fail(B200CONV_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(e_)); break; } }
        CU_BRK(cudaMemsetAsync(p.ring, 0, p.ring_bytes, st));
        CU_BRK(cudaMemsetAsync(p.ypart, 0, p.zmax * m->O * size_t(p.rows) * M * sizeof(float2), st));
        if (p.tickets)
            CU_BRK(cudaMemsetAsync(p.tickets, 0, p.zmax * m->O * sizeof(uint32_t), st));
        if (count == 0)
        {
            CU_BRK(cudaStreamSynchronize(st));
            break;
        }
        std::vector<FoldDesc> fold(count);
        size_t h_row = 0;
        for (size_t r = 0; r < count; ++r)
        {
            const size_t bins = (length[r] + F - 1) >> (rank - 1);
            fold[r].G       = p.G + g_off[r] * M;
            fold[r].head    = nullptr;
            fold[r].h_row   = h_row;
            fold[r].bins    = uint32_t(bins);
            fold[r].pad     = 0;
            h_row          += bins;
        }
        p.rt.resize(count);
        {
            size_t u_at = 0;
            for (size_t i = 0; i < m->I; ++i)
                for (size_t k0 = 0; k0 < leaving[i].size(); k0 += MX_RG, ++u_at)
                    for (uint32_t k = 0; k < units[u_at].nr; ++k)
                    {
                        const size_t r  = leaving[i][k0 + k];
                        units[u_at].G[k] = p.G + g_off[r] * M;
                        p.rt[r]         = MxRoute{ uint32_t(i), uint32_t(output[r]), units[u_at].nq[k],
                                                   uint32_t(u_at), k, units[u_at].G[k], p.G };
                    }
        }
        p.host_units    = units;
        p.nq_cap        = uint32_t(nq_max);
        CU_BRK(cudaMemsetAsync(irdev, 0, rows_total * F * sizeof(float), st));     /* zero padding of every last partition */
        for (size_t r = 0; (r < count) && (rc == B200CONV_OK); ++r)
            CU_BRK(cudaMemcpyAsync(irdev + fold[r].h_row * F, ir[r], length[r] * sizeof(float), cudaMemcpyHostToDevice, st));
        if (rc != B200CONV_OK) break;
        CU_BRK(cudaMemcpyAsync(d_fold, fold.data(), count * sizeof(FoldDesc), cudaMemcpyHostToDevice, st));
        CU_BRK(cudaMemcpyAsync(p.units, units.data(), units.size() * sizeof(MxUnit), cudaMemcpyHostToDevice, st));

        StepArgs a;
        memset(&a, 0, sizeof(a));
        a.tw        = m->tw;
        a.rank      = uint32_t(rank);
        a.splits    = 1;
        a.flags     = STEP_LINEAR_JOBS;
        a.src       = irdev;
        a.dst       = reinterpret_cast<float *>(H);
        CU_BRK(launch_fwd(a, uint32_t(rows_total), st));

        size_t max_bins = 0;
        for (size_t r = 0; r < count; ++r)
            max_bins    = (fold[r].bins > max_bins) ? fold[r].bins : max_bins;
        dim3 grid(uint32_t((F + 255) / 256), uint32_t((max_bins + 1 < 1024) ? max_bins + 1 : 1024),
                  uint32_t((count < 64) ? count : 64));
        k_fold_many<<<grid, 256, 0, st>>>(d_fold, uint32_t(count), H, irdev, uint32_t(F));
        CU_BRK(cudaGetLastError());
        CU_BRK(cudaStreamSynchronize(st));      /* the host arrays above are pageable and about to go */
        #undef CU_BRK
    } while (false);
    if (rc != B200CONV_OK)
        cudaStreamSynchronize(st);
    drop_scratch();
    if (rc != B200CONV_OK)
    {
        mx_plan_free(p, st);
        return rc;
    }

    /* ---- swap in: the old routes, any fade in progress and the history go */
    mx_plan_free(m->plan, st);
    m->plan     = p;
    m->t        = 0;
    return B200CONV_OK;
}

extern "C" int b200conv_mx_set_routes(b200conv_mx_t *m, size_t count, const size_t *input, const size_t *output,
                                      const float *const *ir, const size_t *length)
{
    try { return mx_set_routes_impl(m, count, input, output, ir, length); }
    catch (const std::bad_alloc &) { return fail(B200CONV_ERR_NOMEM, "out of host memory"); }
}

/* New IRs for some routes, keeping the history (header, b200conv_mx_set_irs).  Builds the fade's
 * tables on the host, ingests the IRs on `stream` (k_fwd, then k_fold_delta: G_new and G_new - G_old),
 * and never waits for the device except for the page-locked staging of the previous call. */
static int mx_set_irs_impl(b200conv_mx_t *m, size_t count, const size_t *route, const float *const *ir,
                           const size_t *length, size_t fade, void *stream)
{
    if (m == nullptr)
        return fail(B200CONV_ERR_ARG, "b200conv_mx_set_irs: NULL handle");
    if (count == 0)
        return B200CONV_OK;
    if ((route == nullptr) || (ir == nullptr) || (length == nullptr))
        return fail(B200CONV_ERR_ARG, "b200conv_mx_set_irs: NULL array");
    MxPlan &p = m->plan;
    const size_t F = m->F, M = F, rank = m->rank, I = m->I, O = m->O;

    std::vector<char> seen(p.routes, 0);
    std::vector<uint32_t> bins(count);
    size_t rows_total = 0;
    for (size_t k = 0; k < count; ++k)
    {
        if (route[k] >= p.routes)
            return fail(B200CONV_ERR_ARG, "b200conv_mx_set_irs: route %zu out of range (%zu routes)", route[k], p.routes);
        if (seen[route[k]])
            return fail(B200CONV_ERR_ARG, "b200conv_mx_set_irs: route %zu appears twice", route[k]);
        seen[route[k]] = 1;
        if ((ir[k] == nullptr) || (length[k] == 0))
            return fail(B200CONV_ERR_ARG, "b200conv_mx_set_irs: route %zu: NULL or empty impulse response", route[k]);
        const size_t b = (length[k] >> (rank - 1)) + (((length[k] & (F - 1)) != 0) ? 1 : 0);    /* no wrap */
        if (b + 1 > p.nq_cap)
            return fail(B200CONV_ERR_ARG, "b200conv_mx_set_irs: route %zu: %zu partitions, the ring reaches %u "
                        "(a longer IR needs set_routes)", route[k], b + 1, p.nq_cap);
        bins[k]         = uint32_t(b);
        rows_total     += b;
    }
    if (p.fade.active)
        return fail(B200CONV_ERR_STATE, "b200conv_mx_set_irs: a fade is in progress (%zu samples left)",
                    size_t(p.fade.fade - (m->t - p.fade.t0) * F));

    ENTER_DEVICE(m);
    cudaStream_t st = (stream != nullptr) ? cudaStream_t(stream) : m->stream;

    /* ---- host plan.  Delta output d adds into output omap[d]; one delta route per changed route,
     * grouped by input as set_routes groups the routes; rows of a delta output as those of an output. */
    MxFade f;
    f.fade          = fade;
    f.changed.assign(route, route + count);
    f.nq_new.resize(count);
    std::vector<uint32_t> nd(count);
    for (size_t k = 0; k < count; ++k)
    {
        f.nq_new[k]     = bins[k] + 1;
        nd[k]           = (fade > 0) ? std::max(bins[k] + 1, p.rt[route[k]].nq) : bins[k] + 1;
    }
    std::vector<uint32_t> omap, d_of(O, UINT32_MAX), rank_d(count, 0), fan_d;
    std::vector<MxUnit> dunits;
    if (fade > 0)
    {
        std::vector<size_t> order(count);
        for (size_t k = 0; k < count; ++k)
            order[k]    = k;
        std::sort(order.begin(), order.end(), [&](size_t a, size_t b) { return route[a] < route[b]; });
        for (size_t k : order)
        {
            const uint32_t o = p.rt[route[k]].output;
            if (d_of[o] == UINT32_MAX)
            {
                d_of[o]     = uint32_t(omap.size());
                omap.push_back(o);
                fan_d.push_back(0);
            }
            rank_d[k]   = fan_d[d_of[o]]++;
        }
        f.deltas        = uint32_t(omap.size());
        std::vector<std::vector<size_t>> leaving(I);
        for (size_t k : order)
            leaving[p.rt[route[k]].input].push_back(k);
        for (size_t i = 0; i < I; ++i)
            for (size_t k0 = 0; k0 < leaving[i].size(); k0 += MX_RG)
            {
                MxUnit u;
                memset(&u, 0, sizeof(u));
                u.input         = uint32_t(i);
                u.nr            = uint32_t(std::min<size_t>(MX_RG, leaving[i].size() - k0));
                for (uint32_t s = 0; s < u.nr; ++s)
                {
                    const size_t k  = leaving[i][k0 + s];
                    u.nq[s]         = nd[k];
                    u.row[s]        = (uint32_t(O) + d_of[p.rt[route[k]].output]) * p.rows + rank_d[k] * p.splits;
                    u.nq_max        = std::max(u.nq_max, nd[k]);
                    u.G[s]          = nullptr;          /* the delta spectra: filled in below */
                }
                dunits.push_back(u);
            }
        f.n_units       = p.n_units + uint32_t(dunits.size());
        f.rg            = p.rg;
        for (const MxUnit &u : dunits)
            f.rg            = std::max(f.rg, u.nr);
        const uint32_t TB = uint32_t((M < 1024) ? M : 1024), QB = 1024 / TB;
        f.smem          = size_t(MX_STAGES) * (1 + f.rg) * QB * TB * sizeof(float2) + MX_STAGES * sizeof(uint64_t) + 16;
        const size_t OT = O + f.deltas;
        const size_t per_frame = OT * p.rows * M * sizeof(float2) + ((rank >= 13) ? OT * 2 * F * sizeof(float) : 0) +
                                 f.deltas * F * sizeof(float);
        size_t z        = MX_SCRATCH_BYTES / per_frame;
        z               = std::min<size_t>(z, p.zmax);             /* the ring's spare slots */
        z               = std::min<size_t>(z, (m->job_cap / 2) / (I + OT));    /* >= 1: I + OT <= I + 2 O */
        f.zmax          = uint32_t((z < 1) ? 1 : z);
    }

    /* ---- device memory, stream-ordered; on failure everything allocated here goes again */
    const size_t OT = O + f.deltas;
    float *irdev = nullptr;
    float2 *H = nullptr;
    FoldDeltaDesc *d_desc = nullptr;
    cudaError_t e = cudaSuccess;
    auto alloc = [&](void **ptr, size_t bytes) { if ((e == cudaSuccess) && (bytes > 0)) e = cudaMallocAsync(ptr, bytes, st); };
    f.G_new.assign(count, nullptr);
    for (size_t k = 0; k < count; ++k)
        alloc(reinterpret_cast<void **>(&f.G_new[k]), size_t(bins[k] + 1) * M * sizeof(float2));
    size_t d_rows = 0;
    if (fade > 0)
    {
        for (size_t k = 0; k < count; ++k)
            d_rows         += nd[k];
        alloc(reinterpret_cast<void **>(&f.D), d_rows * M * sizeof(float2));
        alloc(reinterpret_cast<void **>(&f.units), f.n_units * sizeof(MxUnit));
        alloc(reinterpret_cast<void **>(&f.omap), f.deltas * sizeof(uint32_t));
        alloc(reinterpret_cast<void **>(&f.ypart), f.zmax * OT * size_t(p.rows) * M * sizeof(float2));
        alloc(reinterpret_cast<void **>(&f.dout), f.zmax * size_t(f.deltas) * F * sizeof(float));
        if (rank >= 13)
        {
            alloc(reinterpret_cast<void **>(&f.park), f.zmax * OT * 2 * F * sizeof(float));
            alloc(reinterpret_cast<void **>(&f.tickets), f.zmax * OT * sizeof(uint32_t));
        }
    }
    alloc(reinterpret_cast<void **>(&f.units_final), p.n_units * sizeof(MxUnit));
    alloc(reinterpret_cast<void **>(&irdev), rows_total * F * sizeof(float));
    alloc(reinterpret_cast<void **>(&H), rows_total * M * sizeof(float2));
    alloc(reinterpret_cast<void **>(&d_desc), count * sizeof(FoldDeltaDesc));

    /* ---- page-locked staging: padded IR rows, descriptors, the two units tables, omap */
    auto align = [](size_t v) { return (v + 255) & ~size_t(255); };
    const size_t off_desc   = align(rows_total * F * sizeof(float));
    const size_t off_uf     = align(off_desc + count * sizeof(FoldDeltaDesc));
    const size_t off_final  = align(off_uf + f.n_units * sizeof(MxUnit));
    const size_t off_omap   = align(off_final + p.n_units * sizeof(MxUnit));
    const size_t stage      = off_omap + f.deltas * sizeof(uint32_t);
    if ((e == cudaSuccess) && (stage > m->irs_cap))
    {
        if (m->irs_used)
            e = cudaEventSynchronize(m->ev_irs);
        if (e == cudaSuccess)
        {
            const size_t want = std::max(stage, 2 * m->irs_cap);
            if (m->h_irs)
                cudaFreeHost(m->h_irs);
            m->h_irs    = nullptr;
            m->irs_cap  = 0;
            m->irs_used = false;
            e = cudaMallocHost(&m->h_irs, want);
            if (e == cudaSuccess)
                m->irs_cap  = want;
        }
    }
    /* every failure from here on releases what this call allocated (stream-ordered: behind anything
     * of this call already enqueued) and leaves the object as it was */
    auto drop = [&]()
    {
        cudaGetLastError();
        mx_fade_free(f, true, st);
        mx_free_async(irdev, st);
        mx_free_async(H, st);
        mx_free_async(d_desc, st);
    };
    if (e != cudaSuccess)
    {
        drop();
        return fail((e == cudaErrorMemoryAllocation) ? B200CONV_ERR_NOMEM : B200CONV_ERR_CUDA,
                    "b200conv_mx_set_irs: allocation failed: %s", cudaGetErrorString(e));
    }
    if (m->irs_used)
        e = cudaEventSynchronize(m->ev_irs);        /* the previous call's uploads have read the staging */
    if (e != cudaSuccess)
    {
        drop();
        return fail(B200CONV_ERR_CUDA, "b200conv_mx_set_irs: cudaEventSynchronize failed: %s", cudaGetErrorString(e));
    }

    unsigned char *hs   = m->h_irs;
    float *h_ir         = reinterpret_cast<float *>(hs);
    FoldDeltaDesc *h_desc = reinterpret_cast<FoldDeltaDesc *>(hs + off_desc);
    MxUnit *h_uf        = reinterpret_cast<MxUnit *>(hs + off_uf);
    MxUnit *h_final     = reinterpret_cast<MxUnit *>(hs + off_final);
    uint32_t *h_omap    = reinterpret_cast<uint32_t *>(hs + off_omap);
    size_t h_row = 0, d_at = 0;
    uint32_t max_nd = 0;
    f.host_final        = p.host_units;
    for (size_t k = 0; k < count; ++k)
    {
        const MxRoute &r    = p.rt[route[k]];
        float *row          = h_ir + h_row * F;
        memcpy(row, ir[k], length[k] * sizeof(float));
        memset(row + length[k], 0, (size_t(bins[k]) * F - length[k]) * sizeof(float));
        FoldDeltaDesc &d    = h_desc[k];
        d.G         = f.G_new[k];
        d.D         = (fade > 0) ? f.D + d_at * M : nullptr;
        d.G_old     = r.G;
        d.h_row     = h_row;
        d.bins      = bins[k];
        d.nq_old    = r.nq;
        d.nd        = nd[k];
        d.pad       = 0;
        max_nd      = std::max(max_nd, nd[k]);
        h_row      += bins[k];
        d_at       += (fade > 0) ? nd[k] : 0;
        MxUnit &u   = f.host_final[r.unit];
        u.G[r.slot] = f.G_new[k];
        u.nq[r.slot] = f.nq_new[k];
    }
    for (MxUnit &u : f.host_final)
    {
        u.nq_max    = 0;
        for (uint32_t s = 0; s < u.nr; ++s)
            u.nq_max    = std::max(u.nq_max, u.nq[s]);
    }
    if (fade > 0)
    {
        /* delta route k reads D; the delta units list the changed routes in `order` per input */
        std::vector<const float2 *> Dk(count);
        for (size_t k = 0; k < count; ++k)
            Dk[k]       = h_desc[k].D;
        std::vector<std::vector<size_t>> leaving(I);
        std::vector<size_t> order(count);
        for (size_t k = 0; k < count; ++k)
            order[k]    = k;
        std::sort(order.begin(), order.end(), [&](size_t a, size_t b) { return route[a] < route[b]; });
        for (size_t k : order)
            leaving[p.rt[route[k]].input].push_back(k);
        size_t u_at = 0;
        for (size_t i = 0; i < I; ++i)
            for (size_t k0 = 0; k0 < leaving[i].size(); k0 += MX_RG, ++u_at)
                for (uint32_t s = 0; s < dunits[u_at].nr; ++s)
                    dunits[u_at].G[s] = Dk[leaving[i][k0 + s]];
        memcpy(h_uf, p.host_units.data(), p.n_units * sizeof(MxUnit));
        memcpy(h_uf + p.n_units, dunits.data(), dunits.size() * sizeof(MxUnit));
        memcpy(h_omap, omap.data(), omap.size() * sizeof(uint32_t));
    }
    memcpy(h_final, f.host_final.data(), p.n_units * sizeof(MxUnit));

    /* ---- uploads and ingest on `st` */
    int rc = B200CONV_OK;
    do
    {
        #define CU_BRK(call) { cudaError_t e_ = (call); if (e_ != cudaSuccess) { rc = fail(B200CONV_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(e_)); break; } }
        CU_BRK(cudaMemcpyAsync(irdev, h_ir, rows_total * F * sizeof(float), cudaMemcpyHostToDevice, st));
        CU_BRK(cudaMemcpyAsync(d_desc, h_desc, count * sizeof(FoldDeltaDesc), cudaMemcpyHostToDevice, st));
        CU_BRK(cudaMemcpyAsync(f.units_final, h_final, p.n_units * sizeof(MxUnit), cudaMemcpyHostToDevice, st));
        if (fade > 0)
        {
            CU_BRK(cudaMemcpyAsync(f.units, h_uf, f.n_units * sizeof(MxUnit), cudaMemcpyHostToDevice, st));
            CU_BRK(cudaMemcpyAsync(f.omap, h_omap, f.deltas * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
            /* rows no unit writes stay zero (the delta rows' slots change with every call) */
            CU_BRK(cudaMemsetAsync(f.ypart, 0, f.zmax * OT * size_t(p.rows) * M * sizeof(float2), st));
            if (f.tickets)
                CU_BRK(cudaMemsetAsync(f.tickets, 0, f.zmax * OT * sizeof(uint32_t), st));
        }
        CU_BRK(cudaEventRecord(m->ev_irs, st));
        m->irs_used     = true;

        StepArgs a;
        memset(&a, 0, sizeof(a));
        a.tw        = m->tw;
        a.rank      = uint32_t(rank);
        a.splits    = 1;
        a.flags     = STEP_LINEAR_JOBS;
        a.src       = irdev;
        a.dst       = reinterpret_cast<float *>(H);
        CU_BRK(launch_fwd(a, uint32_t(rows_total), st));
        dim3 grid(uint32_t((F + 255) / 256), (max_nd < 1024) ? max_nd : 1024u, uint32_t((count < 64) ? count : 64));
        k_fold_delta<<<grid, 256, 0, st>>>(d_desc, uint32_t(count), H, uint32_t(F));
        CU_BRK(cudaGetLastError());
        #undef CU_BRK
    } while (false);
    if (rc != B200CONV_OK)
    {
        drop();
        return rc;
    }
    mx_free_async(irdev, st);
    mx_free_async(H, st);
    mx_free_async(d_desc, st);

    /* ---- the fade starts with the next call; fade == 0 switches now */
    f.active    = true;
    f.t0        = m->t;
    p.fade      = f;
    if (fade == 0)
        TRY(mx_fade_finish(m, st));
    if (st != m->stream)
    {
        CU(cudaEventRecord(m->ev_last, st));
        m->last_foreign = true;
    }
    return B200CONV_OK;
}

extern "C" int b200conv_mx_set_irs(b200conv_mx_t *m, size_t count, const size_t *route, const float *const *ir,
                                   const size_t *length, size_t fade, void *stream)
{
    try { return mx_set_irs_impl(m, count, route, ir, length, fade, stream); }
    catch (const std::bad_alloc &) { return fail(B200CONV_ERR_NOMEM, "out of host memory"); }
}

/* samples of the fade still to be enqueued: host arithmetic, no device query */
extern "C" size_t b200conv_mx_fade_remaining(const b200conv_mx_t *m)
{
    if ((m == nullptr) || !m->plan.fade.active)
        return 0;
    const MxFade &f = m->plan.fade;
    const uint64_t done = (m->t - f.t0) * m->F;
    return (done >= f.fade) ? 0 : size_t(f.fade - done);
}

extern "C" int b200conv_mx_clear(b200conv_mx_t *m)
{
    if (m == nullptr)
        return fail(B200CONV_ERR_ARG, "b200conv_mx_clear: NULL handle");
    ENTER_DEVICE(m);
    CU(mx_quiesce(m));
    TRY(mx_fade_finish(m, m->stream));      /* a fade in progress ends with the new IRs in place */
    if (m->plan.ring != nullptr)
    {
        CU(cudaMemsetAsync(m->plan.ring, 0, m->plan.ring_bytes, m->stream));
        CU(cudaStreamSynchronize(m->stream));
    }
    m->t        = 0;
    return B200CONV_OK;
}

/* `count` consecutive entries of the job upload ring.  The ring is used in two halves; before a half
 * is written again, the launches that read it last -- all enqueued before the switch to the other
 * half -- must have run: the event recorded at that switch says so.  The host waits only if the
 * device is a whole half ring (MX_GROUP_JOBS jobs) behind. */
static int mx_reserve_jobs(Mx *m, size_t count, cudaStream_t st, size_t *pos)
{
    const size_t half = m->job_cap / 2;
    const size_t cur  = m->job_half;
    if (m->job_pos + count > (cur + 1) * half)
    {
        CU(cudaEventRecord(m->ev_half[cur], st));
        m->half_used[cur] = true;
        const size_t nxt = cur ^ 1;
        if (m->half_used[nxt])
            CU(cudaEventSynchronize(m->ev_half[nxt]));
        m->job_half = nxt;
        m->job_pos  = nxt * half;
    }
    *pos        = m->job_pos;
    m->job_pos += count;
    return B200CONV_OK;
}

/* the attribute is per function and device: raised to the largest footprint any object has launched */
static cudaError_t launch_mx_mac(const MxArgs &x, uint32_t n_units, size_t smem, uint32_t tiles, uint32_t frames,
                                 uint32_t threads, cudaStream_t st)
{
    static size_t attr_smem[MAX_DEVICES] = { 0 };
    const int dev = current_device();
    if (smem > attr_smem[dev])
    {
        cudaError_t e = cudaFuncSetAttribute(k_mx_mac, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
        if (e != cudaSuccess)
            return e;
        attr_smem[dev] = smem;
    }
    return launch_k(k_mx_mac, dim3(n_units * x.splits, tiles, frames), dim3(threads), smem, st, true, x);
}

static int mx_process_device_impl(b200conv_mx_t *m, float *dst, size_t dst_stride, const float *src, size_t src_stride,
                                  size_t count, void *stream)
{
    if (m == nullptr)
        return fail(B200CONV_ERR_ARG, "b200conv_mx_process_device: NULL handle");
    if ((count % m->F) != 0)
        return fail(B200CONV_ERR_ARG, "b200conv_mx_process_device: count %zu is not a multiple of the frame size %zu",
                    count, m->F);
    if (count == 0)
        return B200CONV_OK;
    if ((dst == nullptr) || (src == nullptr) || ((m->I > 1) && (src_stride < count)) ||
        ((m->O > 1) && (dst_stride < count)))
        return fail(B200CONV_ERR_ARG, "b200conv_mx_process_device: bad buffers");
    ENTER_DEVICE(m);
    cudaStream_t st = (stream != nullptr) ? cudaStream_t(stream) : m->stream;
    const MxPlan &p = m->plan;
    const size_t F = m->F, M = F, I = m->I, O = m->O;

    if (p.routes == 0)
        CU(cudaMemset2DAsync(dst, ((O > 1) ? dst_stride : count) * sizeof(float), 0, count * sizeof(float), O, st));
    else
    {
        const size_t frames = count / F;
        const uint32_t TB = uint32_t((M < 1024) ? M : 1024);
        for (size_t f0 = 0; f0 < frames; )
        {
            /* during a fade: the delta outputs follow the real ones (outputs O .. O + deltas - 1) */
            const MxFade &fd    = p.fade;
            const bool fading   = fd.active;
            const size_t OT     = O + (fading ? fd.deltas : 0);
            const uint32_t zcap = fading ? fd.zmax : p.zmax;
            const uint32_t Z = uint32_t((frames - f0 < zcap) ? frames - f0 : zcap);
            size_t pos = 0;
            TRY(mx_reserve_jobs(m, size_t(Z) * (I + OT), st, &pos));
            Job *jf = m->h_jobs + pos, *ji = jf + size_t(Z) * I;
            memset(jf, 0, size_t(Z) * (I + OT) * sizeof(Job));
            for (uint32_t z = 0; z < Z; ++z)
            {
                const uint64_t t    = m->t + z;
                const uint32_t tm   = uint32_t(t % p.S);
                const uint32_t slot = (tm == 0) ? 0 : p.S - tm;
                for (size_t i = 0; i < I; ++i)
                {
                    Job &j      = jf[size_t(z) * I + i];
                    j.src       = src + i * src_stride + (f0 + z) * F;
                    j.spec      = p.ring + (i * p.S + slot) * M;
                }
                for (size_t o = 0; o < O; ++o)
                    ji[size_t(z) * OT + o].dst = dst + o * dst_stride + (f0 + z) * F;
                for (size_t d = 0; d < OT - O; ++d)
                    ji[size_t(z) * OT + O + d].dst = fd.dout + (size_t(z) * fd.deltas + d) * F;
            }
            CU(cudaMemcpyAsync(m->d_jobs + pos, jf, size_t(Z) * (I + OT) * sizeof(Job), cudaMemcpyHostToDevice, st));

            StepArgs a;
            memset(&a, 0, sizeof(a));
            a.tw        = m->tw;
            a.rank      = uint32_t(m->rank);
            a.splits    = 1;
            a.jobs      = m->d_jobs + pos;
            CU(launch_fwd(a, Z * uint32_t(I), st, false));

            MxArgs x;
            memset(&x, 0, sizeof(x));
            x.units     = fading ? fd.units : p.units;
            x.ring      = p.ring;
            x.ypart     = fading ? fd.ypart : p.ypart;
            x.t_base    = m->t;
            x.S         = p.S;
            x.rank      = uint32_t(m->rank);
            x.splits    = p.splits;
            x.rows      = p.rows;
            x.outputs   = uint32_t(OT);
            x.TB        = TB;
            x.QB        = 1024 / TB;
            x.rg        = fading ? fd.rg : p.rg;
            CU(launch_mx_mac(x, fading ? fd.n_units : p.n_units, fading ? fd.smem : p.smem, uint32_t(M / TB), Z,
                             TB / (2 * MAC_VPT), st));

            a.jobs      = m->d_jobs + pos + size_t(Z) * I;
            a.ypart     = x.ypart;
            a.rows      = p.rows;
            a.splits    = p.rows;
            a.park      = fading ? fd.park : p.park;
            CU(launch_inv(a, Z * uint32_t(OT), st, true, fading ? fd.tickets : p.tickets));
            if (fading)
            {
                dim3 grid(uint32_t((F + 255) / 256), fd.deltas, Z);
                k_mx_blend<<<grid, 256, 0, st>>>(dst + f0 * F, dst_stride, fd.dout, fd.omap, fd.deltas, uint32_t(F),
                                                 (m->t - fd.t0) * F, fd.fade);
                CU(cudaGetLastError());
            }
            m->t       += Z;
            f0         += Z;
            if (fading && ((m->t - fd.t0) * F >= fd.fade))
                TRY(mx_fade_finish(m, st));
        }
    }
    if (st != m->stream)
    {
        CU(cudaEventRecord(m->ev_last, st));
        m->last_foreign = true;
    }
    return B200CONV_OK;
}

extern "C" int b200conv_mx_process_device(b200conv_mx_t *m, float *dst, size_t dst_stride, const float *src,
                                          size_t src_stride, size_t count, void *stream)
{
    try { return mx_process_device_impl(m, dst, dst_stride, src, src_stride, count, stream); }
    catch (const std::bad_alloc &) { return fail(B200CONV_ERR_NOMEM, "out of host memory"); }
}

/* Host matrices [inputs][src_stride] -> [outputs][dst_stride]; synchronous. */
extern "C" int b200conv_mx_process_planar(b200conv_mx_t *m, float *dst, size_t dst_stride, const float *src,
                                          size_t src_stride, size_t count)
{
    if (m == nullptr)
        return fail(B200CONV_ERR_ARG, "b200conv_mx_process_planar: NULL handle");
    if ((count % m->F) != 0)
        return fail(B200CONV_ERR_ARG, "b200conv_mx_process_planar: count %zu is not a multiple of the frame size %zu",
                    count, m->F);
    if (count == 0)
        return B200CONV_OK;
    if ((dst == nullptr) || (src == nullptr) || ((m->I > 1) && (src_stride < count)) ||
        ((m->O > 1) && (dst_stride < count)))
        return fail(B200CONV_ERR_ARG, "b200conv_mx_process_planar: bad buffers");
    ENTER_DEVICE(m);
    if (m->I == 1)  src_stride = count;             /* one row: any pitch */
    if (m->O == 1)  dst_stride = count;
    const size_t rows = (m->I > m->O) ? m->I : m->O;
    size_t cap = ((size_t(1) << 24) / rows) / m->F * m->F;
    if (cap < m->F)     cap = m->F;
    for (size_t done = 0; done < count; )
    {
        const size_t c = (count - done < cap) ? count - done : cap;
        if (c > m->stage_cols)
        {
            CU(mx_quiesce(m));
            if (m->sd_in)   cudaFree(m->sd_in);
            if (m->sd_out)  cudaFree(m->sd_out);
            m->sd_in = m->sd_out = nullptr;
            m->stage_cols = 0;
            CU(cudaMalloc(&m->sd_in, m->I * c * sizeof(float)));
            CU(cudaMalloc(&m->sd_out, m->O * c * sizeof(float)));
            m->stage_cols = c;
        }
        CU(cudaMemcpy2DAsync(m->sd_in, c * sizeof(float), src + done, src_stride * sizeof(float), c * sizeof(float), m->I,
                             cudaMemcpyHostToDevice, m->stream));
        TRY(b200conv_mx_process_device(m, m->sd_out, c, m->sd_in, c, c, m->stream));
        CU(cudaMemcpy2DAsync(dst + done, dst_stride * sizeof(float), m->sd_out, c * sizeof(float), c * sizeof(float), m->O,
                             cudaMemcpyDeviceToHost, m->stream));
        CU(cudaStreamSynchronize(m->stream));
        done += c;
    }
    return B200CONV_OK;
}

extern "C" int b200conv_mx_sync(b200conv_mx_t *m)
{
    if (m == nullptr)
        return fail(B200CONV_ERR_ARG, "b200conv_mx_sync: NULL handle");
    ENTER_DEVICE(m);
    CU(mx_quiesce(m));
    return B200CONV_OK;
}

extern "C" void *b200conv_mx_stream(b200conv_mx_t *m)              { return (m != nullptr) ? (void *)m->stream : nullptr; }
extern "C" size_t b200conv_mx_inputs(const b200conv_mx_t *m)        { return (m != nullptr) ? m->I : 0; }
extern "C" size_t b200conv_mx_outputs(const b200conv_mx_t *m)       { return (m != nullptr) ? m->O : 0; }
extern "C" size_t b200conv_mx_rank(const b200conv_mx_t *m)          { return (m != nullptr) ? m->rank : 0; }
extern "C" size_t b200conv_mx_frame_size(const b200conv_mx_t *m)    { return (m != nullptr) ? m->F : 0; }
extern "C" size_t b200conv_mx_routes(const b200conv_mx_t *m)        { return (m != nullptr) ? m->plan.routes : 0; }

#endif /* B200CONV_MATRIX_HOST_CUH_ */

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
 */
#ifndef B200CONV_MATRIX_HOST_CUH_
#define B200CONV_MATRIX_HOST_CUH_

static const size_t   MX_MAX_IO         = 4096;                 /* inputs, outputs per object */
static const uint32_t MX_GROUP_FRAMES   = 32;                   /* frames per launch group (bounds the ring's spare slots) */
static const size_t   MX_GROUP_JOBS     = size_t(1) << 13;      /* transform jobs per launch group */
static const size_t   MX_SCRATCH_BYTES  = size_t(256) << 20;    /* partial rows + half-frame scratch of one launch group */

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
    size_t      ring_bytes  = 0;
    size_t      smem        = 0;
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
};

typedef b200conv_mx Mx;

static void mx_plan_free(MxPlan &p)
{
    if (p.G)        cudaFree(p.G);
    if (p.ring)     cudaFree(p.ring);
    if (p.ypart)    cudaFree(p.ypart);
    if (p.park)     cudaFree(p.park);
    if (p.tickets)  cudaFree(p.tickets);
    if (p.units)    cudaFree(p.units);
    p = MxPlan();
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
    if (m->stream)  mx_quiesce(m);
    mx_plan_free(m->plan);
    if (m->tw)      cudaFree(m->tw);
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
    /* two halves, each holding the jobs of the largest launch group */
    m->job_cap  = 2 * MX_GROUP_JOBS;

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
        const size_t bins = (length[r] + F - 1) >> (rank - 1);
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
        alloc(reinterpret_cast<void **>(&p.G), g_rows * M * sizeof(float2));
        alloc(reinterpret_cast<void **>(&p.units), units.size() * sizeof(MxUnit));
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
        mx_plan_free(p);
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
        {
            size_t u_at = 0;
            for (size_t i = 0; i < m->I; ++i)
                for (size_t k0 = 0; k0 < leaving[i].size(); k0 += MX_RG, ++u_at)
                    for (uint32_t k = 0; k < units[u_at].nr; ++k)
                        units[u_at].G[k] = p.G + g_off[leaving[i][k0 + k]] * M;
        }
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
        mx_plan_free(p);
        return rc;
    }

    /* ---- swap in: the old routes and history go */
    mx_plan_free(m->plan);
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

extern "C" int b200conv_mx_clear(b200conv_mx_t *m)
{
    if (m == nullptr)
        return fail(B200CONV_ERR_ARG, "b200conv_mx_clear: NULL handle");
    ENTER_DEVICE(m);
    CU(mx_quiesce(m));
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
static cudaError_t launch_mx_mac(const MxArgs &x, const MxPlan &p, uint32_t tiles, uint32_t frames, uint32_t threads,
                                 cudaStream_t st)
{
    static size_t attr_smem[MAX_DEVICES] = { 0 };
    const int dev = current_device();
    if (p.smem > attr_smem[dev])
    {
        cudaError_t e = cudaFuncSetAttribute(k_mx_mac, cudaFuncAttributeMaxDynamicSharedMemorySize, int(p.smem));
        if (e != cudaSuccess)
            return e;
        attr_smem[dev] = p.smem;
    }
    return launch_k(k_mx_mac, dim3(p.n_units * p.splits, tiles, frames), dim3(threads), p.smem, st, true, x);
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
            const uint32_t Z = uint32_t((frames - f0 < p.zmax) ? frames - f0 : p.zmax);
            size_t pos = 0;
            TRY(mx_reserve_jobs(m, size_t(Z) * (I + O), st, &pos));
            Job *jf = m->h_jobs + pos, *ji = jf + size_t(Z) * I;
            memset(jf, 0, size_t(Z) * (I + O) * sizeof(Job));
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
                    ji[size_t(z) * O + o].dst = dst + o * dst_stride + (f0 + z) * F;
            }
            CU(cudaMemcpyAsync(m->d_jobs + pos, jf, size_t(Z) * (I + O) * sizeof(Job), cudaMemcpyHostToDevice, st));

            StepArgs a;
            memset(&a, 0, sizeof(a));
            a.tw        = m->tw;
            a.rank      = uint32_t(m->rank);
            a.splits    = 1;
            a.jobs      = m->d_jobs + pos;
            CU(launch_fwd(a, Z * uint32_t(I), st, false));

            MxArgs x;
            memset(&x, 0, sizeof(x));
            x.units     = p.units;
            x.ring      = p.ring;
            x.ypart     = p.ypart;
            x.t_base    = m->t;
            x.S         = p.S;
            x.rank      = uint32_t(m->rank);
            x.splits    = p.splits;
            x.rows      = p.rows;
            x.outputs   = uint32_t(O);
            x.TB        = TB;
            x.QB        = 1024 / TB;
            x.rg        = p.rg;
            CU(launch_mx_mac(x, p, uint32_t(M / TB), Z, TB / (2 * MAC_VPT), st));

            a.jobs      = m->d_jobs + pos + size_t(Z) * I;
            a.ypart     = p.ypart;
            a.rows      = p.rows;
            a.splits    = p.rows;
            a.park      = p.park;
            CU(launch_inv(a, Z * uint32_t(O), st, true, p.tickets));
            m->t       += Z;
            f0         += Z;
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

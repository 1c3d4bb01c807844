/*
 * spectral_host.cuh -- host side and C ABI (b200conv_sp_*) of the batched SpectralProcessor
 * (scope-table row f4; included by engine.cu after spectral.cuh).
 *
 * Bookkeeping follows lsp::dspu::SpectralProcessor (reference src/main/util/SpectralProcessor.cpp):
 * init :58-75, update_settings :107-125 (buffers cleared, nOffset = size_t(N * (fPhase * 0.5f))),
 * set_phase :127-131 (clamped to [0, 1]), set_rank :133-141 (ignored when equal or above the
 * maximum), process :143-199, remaining :241-245, reset :247-257 (clears the buffers, keeps nOffset,
 * does nothing while an update is pending), latency() = 2^rank (SpectralProcessor.h).
 */
#ifndef B200CONV_SPECTRAL_HOST_CUH_
#define B200CONV_SPECTRAL_HOST_CUH_

static const size_t SP_RANK_MIN = 7, SP_RANK_MAX = 15;      /* transform rank + 1 must be one of the engine's 8..16 */

struct b200conv_sp
{
    int                     device      = 0;
    int                     sm_count    = 148;
    size_t                  n           = 0;
    size_t                  max_rank    = 0, rank = 0;
    cudaStream_t            stream      = nullptr;
    float2                 *tw[B200CONV_RANK_MAX + 1] = { nullptr };    /* by transform rank (= rank + 1) */
    float                  *d_wnd       = nullptr;      /* [2^max_rank] window of the CURRENT rank            */
    float                  *d_in = nullptr, *d_out = nullptr;           /* [n][2^max_rank] each               */
    float2                 *d_table     = nullptr;      /* [n][2^(max_rank-1) + 1] folded tables              */
    uint8_t                *d_bound     = nullptr;
    uint32_t               *d_off       = nullptr;
    std::vector<uint32_t>   h_off;
    std::vector<float>      phase;
    std::vector<uint8_t>    dirty, bound;               /* bUpdate per instance; SP_UNBOUND / _TABLE / _FUNCTION */
    bool                    wnd_dirty   = true, bound_dirty = true;
    float                  *s_in = nullptr, *s_out = nullptr, *sd_in = nullptr, *sd_out = nullptr;   /* host staging */
    size_t                  stage_floats = 0;
    /* the spectral function (b200conv_sp_set_function) and what its sub-calls need */
    b200conv_sp_func_t      fn          = nullptr;
    void                   *fn_user     = nullptr;
    bool                    in_fn       = false;        /* the function is running: the object refuses calls */
    float2                 *d_spectra   = nullptr;      /* [frames][2^rank], stream-ordered allocation        */
    size_t                  spectra_cap = 0;            /* bytes                                              */
    unsigned char          *d_tab       = nullptr;      /* frame table + SpFnInst list, stream-ordered         */
    size_t                  tab_cap     = 0;            /* bytes                                              */
    unsigned char          *h_tab[2]    = { nullptr, nullptr };     /* page-locked staging, used in turn      */
    size_t                  h_tab_cap[2] = { 0, 0 };
    cudaEvent_t             ev_tab[2]   = { nullptr, nullptr };     /* the upload from h_tab[i] has run       */
    bool                    tab_used[2] = { false, false };
    int                     tab_cur     = 0;
};

typedef b200conv_sp Sp;

enum SpKernel { SP_K_SP = 0, SP_K_FWD = 1, SP_K_INV = 2 };

template <int RANKP, int K>
static cudaError_t launch_sp_k(const SpArgs &a, uint32_t grid, cudaStream_t st)
{
    using S = SpCfg<RANKP>;
    constexpr auto kernel = (K == SP_K_SP) ? k_sp<RANKP> : (K == SP_K_FWD) ? k_sp_fwd<RANKP> : k_sp_inv<RANKP>;
    static bool attr_set[MAX_DEVICES] = { false };
    int dev = current_device();
    if ((!attr_set[dev]) && (S::SMEM > 48 * 1024))
    {
        cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(S::SMEM));
        if (e != cudaSuccess)
            return e;
    }
    attr_set[dev] = true;
    kernel<<<grid, S::C::T, S::SMEM, st>>>(a);
    return cudaGetLastError();
}

template <int RANKP>
static cudaError_t launch_sp_r(const SpArgs &a, SpKernel k, uint32_t grid, cudaStream_t st)
{
    switch (k)
    {
        case SP_K_SP:   return launch_sp_k<RANKP, SP_K_SP>(a, grid, st);
        case SP_K_FWD:  return launch_sp_k<RANKP, SP_K_FWD>(a, grid, st);
        default:        return launch_sp_k<RANKP, SP_K_INV>(a, grid, st);
    }
}

static cudaError_t launch_sp(const SpArgs &a, SpKernel k, size_t rank, uint32_t grid, cudaStream_t st)
{
    switch (rank + 1)
    {
        case 8:  return launch_sp_r<8>(a, k, grid, st);
        case 9:  return launch_sp_r<9>(a, k, grid, st);
        case 10: return launch_sp_r<10>(a, k, grid, st);
        case 11: return launch_sp_r<11>(a, k, grid, st);
        case 12: return launch_sp_r<12>(a, k, grid, st);
        case 13: return launch_sp_r<13>(a, k, grid, st);
        case 14: return launch_sp_r<14>(a, k, grid, st);
        case 15: return launch_sp_r<15>(a, k, grid, st);
        case 16: return launch_sp_r<16>(a, k, grid, st);
        default: return cudaErrorInvalidValue;
    }
}

/* Every entry point that changes the object refuses to run from inside its spectral function. */
#define SP_NOT_IN_FN(s, what)                                                                   \
    if ((s)->in_fn)                                                                             \
        return fail(B200CONV_ERR_STATE, "%s: called from inside the object's spectral function", what)

extern "C" void b200conv_sp_free(b200conv_sp_t *s)
{
    if (s == nullptr)
        return;
    DeviceScope device_scope_(s->device);
    if (s->stream)  cudaStreamSynchronize(s->stream);
    for (float2 *t : s->tw)
        if (t) cudaFree(t);
    if (s->d_wnd)   cudaFree(s->d_wnd);
    if (s->d_in)    cudaFree(s->d_in);
    if (s->d_out)   cudaFree(s->d_out);
    if (s->d_table) cudaFree(s->d_table);
    if (s->d_bound) cudaFree(s->d_bound);
    if (s->d_off)   cudaFree(s->d_off);
    if (s->s_in)    cudaFreeHost(s->s_in);
    if (s->s_out)   cudaFreeHost(s->s_out);
    if (s->sd_in)   cudaFree(s->sd_in);
    if (s->sd_out)  cudaFree(s->sd_out);
    if (s->stream)
    {
        if (s->d_spectra)   cudaFreeAsync(s->d_spectra, s->stream);
        if (s->d_tab)       cudaFreeAsync(s->d_tab, s->stream);
        cudaStreamSynchronize(s->stream);
    }
    for (int i = 0; i < 2; ++i)
    {
        if (s->h_tab[i])    cudaFreeHost(s->h_tab[i]);
        if (s->ev_tab[i])   cudaEventDestroy(s->ev_tab[i]);
    }
    if (s->stream)  cudaStreamDestroy(s->stream);
    delete s;
}

static int sp_create_impl(b200conv_sp_t **out, int device, size_t instances, size_t max_rank)
{
    if ((out == nullptr) || (instances == 0) || (instances > (size_t(1) << 20)) ||
        (max_rank < SP_RANK_MIN) || (max_rank > SP_RANK_MAX))
        return fail(B200CONV_ERR_ARG, "b200conv_sp_create: bad arguments (ranks %zu..%zu)", SP_RANK_MIN, SP_RANK_MAX);
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if ((e != cudaSuccess) || (count == 0))
        return fail(B200CONV_ERR_CUDA, "no CUDA device available (%s); this engine has no CPU fallback", cudaGetErrorString(e));
    if (device < 0)
        CU(cudaGetDevice(&device));
    if (device >= count)
        return fail(B200CONV_ERR_ARG, "device %d out of range (%d devices)", device, count);

    Sp *s = new (std::nothrow) Sp();
    if (s == nullptr)
        return fail(B200CONV_ERR_NOMEM, "out of host memory");
    s->device   = device;
    s->n        = instances;
    s->max_rank = s->rank = max_rank;               /* SpectralProcessor.cpp:60-61 */
    s->h_off.assign(instances, 0);
    s->phase.assign(instances, 0.0f);
    s->dirty.assign(instances, 1);                  /* bUpdate = true (:63) */
    s->bound.assign(instances, 0);

    ENTER_DEVICE(s);
    const size_t N = size_t(1) << max_rank;
    int rc = B200CONV_OK;
    do
    {
        cudaDeviceProp prop;
        if (cudaGetDeviceProperties(&prop, device) == cudaSuccess)
            s->sm_count = prop.multiProcessorCount;
        #define CU_BRK(call) { cudaError_t e_ = (call); if (e_ != cudaSuccess) { rc = fail((e_ == cudaErrorMemoryAllocation) ? B200CONV_ERR_NOMEM : B200CONV_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(e_)); break; } }
        CU_BRK(cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking));
        CU_BRK(cudaEventCreateWithFlags(&s->ev_tab[0], cudaEventDisableTiming));
        CU_BRK(cudaEventCreateWithFlags(&s->ev_tab[1], cudaEventDisableTiming));
        CU_BRK(cudaMalloc(&s->d_wnd, N * sizeof(float)));
        CU_BRK(cudaMalloc(&s->d_in, instances * N * sizeof(float)));
        CU_BRK(cudaMalloc(&s->d_out, instances * N * sizeof(float)));
        CU_BRK(cudaMalloc(&s->d_table, instances * (N / 2 + 1) * sizeof(float2)));
        CU_BRK(cudaMalloc(&s->d_bound, instances));
        CU_BRK(cudaMalloc(&s->d_off, instances * sizeof(uint32_t)));
        CU_BRK(cudaMemset(s->d_bound, 0, instances));
        #undef CU_BRK
    } while (false);
    if (rc != B200CONV_OK)
    {
        std::string keep = g_last_error;
        b200conv_sp_free(s);
        g_last_error = keep;
        return rc;
    }
    *out = s;
    return B200CONV_OK;
}

extern "C" int b200conv_sp_create(b200conv_sp_t **out, int device, size_t instances, size_t max_rank)
{
    try { return sp_create_impl(out, device, instances, max_rank); }
    catch (const std::bad_alloc &) { return fail(B200CONV_ERR_NOMEM, "out of host memory"); }
}

extern "C" int b200conv_sp_set_rank(b200conv_sp_t *s, size_t rank)
{
    if (s == nullptr)
        return fail(B200CONV_ERR_ARG, "b200conv_sp_set_rank: NULL handle");
    SP_NOT_IN_FN(s, "b200conv_sp_set_rank");
    if ((rank == s->rank) || (rank > s->max_rank))          /* SpectralProcessor.cpp:135-136 */
        return B200CONV_OK;
    if (rank < SP_RANK_MIN)
        return fail(B200CONV_ERR_ARG, "b200conv_sp_set_rank: ranks below %zu are not supported", SP_RANK_MIN);
    s->rank         = rank;
    s->wnd_dirty    = true;
    for (size_t i = 0; i < s->n; ++i)
    {
        s->dirty[i]     = 1;                                /* bUpdate = true (:139) */
        if (s->bound[i] == SP_TABLE)
            s->bound[i]     = SP_UNBOUND;                   /* tables are rank-specific: bind again; pFunc stays */
    }
    s->bound_dirty  = true;
    return B200CONV_OK;
}

extern "C" int b200conv_sp_set_phase(b200conv_sp_t *s, size_t idx, float phase)
{
    if ((s == nullptr) || (idx >= s->n))
        return fail(B200CONV_ERR_ARG, "b200conv_sp_set_phase: bad handle or index");
    SP_NOT_IN_FN(s, "b200conv_sp_set_phase");
    s->phase[idx]   = (phase < 0.0f) ? 0.0f : ((phase > 1.0f) ? 1.0f : phase);      /* lsp_limit, :129 */
    s->dirty[idx]   = 1;
    return B200CONV_OK;
}

/* kind 0: unbind; 1: `table` = 2^rank packed complex bins; 2: `table` = 2^rank real gains;
 * 3: the object's spectral function */
static int sp_bind(b200conv_sp_t *s, size_t idx, int kind, const float *table)
{
    if ((s == nullptr) || (idx >= s->n) || (((kind == 1) || (kind == 2)) && (table == nullptr)))
        return fail(B200CONV_ERR_ARG, "b200conv_sp_bind: bad arguments");
    SP_NOT_IN_FN(s, "b200conv_sp_bind");
    ENTER_DEVICE(s);
    if ((kind == 0) || (kind == 3))
    {
        if ((kind == 3) && (s->fn == nullptr))
            return fail(B200CONV_ERR_STATE, "b200conv_sp_bind_function: no spectral function set");
        s->bound[idx]   = (kind == 3) ? SP_FUNCTION : SP_UNBOUND;
        s->bound_dirty  = true;
        return B200CONV_OK;
    }
    /* Re(IFFT(X H)) for real input = the half-spectrum product with (H[k] + conj(H[N - k])) / 2 */
    const size_t N = size_t(1) << s->rank, P = N / 2;
    std::vector<float2> folded(P + 1);
    for (size_t k = 0; k <= P; ++k)
    {
        const size_t km = (N - k) % N;
        if (kind == 1)
            folded[k]   = make_float2(0.5f * (table[2 * k] + table[2 * km]), 0.5f * (table[2 * k + 1] - table[2 * km + 1]));
        else
            folded[k]   = make_float2(0.5f * (table[k] + table[km]), 0.0f);
    }
    CU(cudaStreamSynchronize(s->stream));
    CU(cudaMemcpy(s->d_table + idx * (P + 1), folded.data(), (P + 1) * sizeof(float2), cudaMemcpyHostToDevice));
    s->bound[idx]   = SP_TABLE;
    s->bound_dirty  = true;
    return B200CONV_OK;
}

extern "C" int b200conv_sp_bind_complex(b200conv_sp_t *s, size_t idx, const float *table)
{
    try { return sp_bind(s, idx, 1, table); }
    catch (const std::bad_alloc &) { return fail(B200CONV_ERR_NOMEM, "out of host memory"); }
}

extern "C" int b200conv_sp_bind_gain(b200conv_sp_t *s, size_t idx, const float *gain)
{
    try { return sp_bind(s, idx, 2, gain); }
    catch (const std::bad_alloc &) { return fail(B200CONV_ERR_NOMEM, "out of host memory"); }
}

extern "C" int b200conv_sp_unbind(b200conv_sp_t *s, size_t idx)
{
    return sp_bind(s, idx, 0, nullptr);
}

extern "C" int b200conv_sp_bind_function(b200conv_sp_t *s, size_t idx)
{
    return sp_bind(s, idx, 3, nullptr);
}

extern "C" int b200conv_sp_set_function(b200conv_sp_t *s, b200conv_sp_func_t fn, void *user)
{
    if (s == nullptr)
        return fail(B200CONV_ERR_ARG, "b200conv_sp_set_function: NULL handle");
    SP_NOT_IN_FN(s, "b200conv_sp_set_function");
    if (fn == nullptr)
        for (size_t i = 0; i < s->n; ++i)
            if (s->bound[i] == SP_FUNCTION)
                return fail(B200CONV_ERR_STATE, "b200conv_sp_set_function: instance %zu is bound to the function", i);
    s->fn           = fn;
    s->fn_user      = user;
    return B200CONV_OK;
}

/* SpectralProcessor::update_settings for the instances that asked for it (:107-125), then the
 * tables the kernel reads. */
static int sp_commit(Sp *s, cudaStream_t st)
{
    const size_t N = size_t(1) << s->rank;
    bool any = false;
    for (size_t i = 0; i < s->n; ++i)
    {
        if (!s->dirty[i])
            continue;
        any             = true;
        /* the buffers of the instance are laid out with the CURRENT rank's pitch: a rank change marks
         * every instance, so the whole arrays are cleared below */
        s->h_off[i]     = uint32_t(size_t(float(N) * (s->phase[i] * 0.5f)));        /* :123, fp32 */
    }
    if (any)
    {
        bool all = true;
        for (size_t i = 0; i < s->n; ++i)
            all             = all && (s->dirty[i] != 0);
        if (all)
        {
            CU(cudaMemsetAsync(s->d_in, 0, s->n * N * sizeof(float), st));
            CU(cudaMemsetAsync(s->d_out, 0, s->n * N * sizeof(float), st));
        }
        else
            for (size_t i = 0; i < s->n; ++i)
                if (s->dirty[i])
                {
                    CU(cudaMemsetAsync(s->d_in + i * N, 0, N * sizeof(float), st));
                    CU(cudaMemsetAsync(s->d_out + i * N, 0, N * sizeof(float), st));
                }
        CU(cudaMemcpyAsync(s->d_off, s->h_off.data(), s->n * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
        for (size_t i = 0; i < s->n; ++i)
            s->dirty[i]     = 0;
    }
    if (s->wnd_dirty)
    {
        /* windows::cosine (reference src/main/misc/windows.cpp:238-246): f = M_PI / n in fp32, sinf(f * i) */
        std::vector<float> w(N);
        const float f   = float(M_PI / double(N));
        for (size_t i = 0; i < N; ++i)
            w[i]            = sinf(f * float(i));
        CU(cudaMemcpyAsync(s->d_wnd, w.data(), N * sizeof(float), cudaMemcpyHostToDevice, st));
        CU(cudaStreamSynchronize(st));          /* `w` is pageable and about to go out of scope */
        s->wnd_dirty    = false;
    }
    if (s->bound_dirty)
    {
        CU(cudaMemcpyAsync(s->d_bound, s->bound.data(), s->n, cudaMemcpyHostToDevice, st));
        s->bound_dirty  = false;
    }
    if (s->tw[s->rank + 1] == nullptr)
        TRY(make_twiddles(uint32_t(s->rank + 1), &s->tw[s->rank + 1]));
    return B200CONV_OK;
}

/* nOffset after `count` samples from `off` (the kernels' loop, :154-198, F = N / 2): every time the
 * offset reaches F with samples left it restarts at 0 */
static uint32_t sp_advance(uint32_t off, uint64_t count, uint32_t F)
{
    uint64_t total  = uint64_t(off) + count;
    if (off >= F)
        total           = count;            /* a transform precedes the first sample */
    return (total <= F) ? uint32_t(total) : uint32_t((total - 1) % F + 1);
}

/* Samples of a sub-call of B function-bound instances: L = P * max(1, floor(2^25 / (B * N))). */
static size_t sp_fn_span(size_t rank, size_t B)
{
    const size_t N = size_t(1) << rank;
    const size_t q = (size_t(1) << 25) / (B * N);
    return (N / 2) * ((q > 1) ? q : 1);
}

/* `bytes` of stream-ordered device memory at *p, grown (never shrunk) on the call's stream */
static cudaError_t sp_grow_async(void **p, size_t *cap, size_t bytes, cudaStream_t st)
{
    if (bytes <= *cap)
        return cudaSuccess;
    if (*p)
        cudaFreeAsync(*p, st);
    *p      = nullptr;
    *cap    = 0;
    cudaError_t e = cudaMallocAsync(p, bytes, st);
    if (e == cudaSuccess)
        *cap    = bytes;
    return e;
}

/* The function-bound instances `fi` over one call: per sub-call, k_sp_fwd, the spectral function and
 * k_sp_inv.  `a` is the call's launch (all rows from sample 0); `base` is the position of the call's
 * first sample in the caller's process call.  Leaves h_off of these instances untouched. */
static int sp_run_function(Sp *s, const SpArgs &call, const std::vector<uint32_t> &fi, size_t count, size_t base,
                           uint32_t grid, cudaStream_t st)
{
    const uint32_t F    = uint32_t(1) << (s->rank - 1);
    const size_t N      = size_t(2) * F;
    const size_t B      = fi.size();
    const size_t L      = sp_fn_span(s->rank, B);
    std::vector<uint32_t> off(B);
    for (size_t j = 0; j < B; ++j)
        off[j]              = s->h_off[fi[j]];

    for (size_t s0 = 0; s0 < count; )
    {
        /* sub-calls start at multiples of L of the caller's call */
        const size_t len    = std::min(L - (base + s0) % L, count - s0);
        size_t nf           = 0;
        for (size_t j = 0; j < B; ++j)
        {
            const size_t p0     = (off[j] >= F) ? 0 : F - off[j];
            nf                 += (p0 < len) ? (len - 1 - p0) / F + 1 : 0;
        }
        const size_t fn_at  = (nf * sizeof(b200conv_sp_frame_t) + 15) & ~size_t(15);
        const size_t bytes  = fn_at + B * sizeof(SpFnInst);

        /* page-locked staging, two in turn: wait only while the upload from this one still reads it */
        const int h         = s->tab_cur;
        if (s->tab_used[h])
            CU(cudaEventSynchronize(s->ev_tab[h]));
        s->tab_used[h]      = false;
        if (bytes > s->h_tab_cap[h])
        {
            if (s->h_tab[h])
                cudaFreeHost(s->h_tab[h]);
            s->h_tab[h]         = nullptr;
            s->h_tab_cap[h]     = 0;
            CU(cudaMallocHost(reinterpret_cast<void **>(&s->h_tab[h]), bytes));
            s->h_tab_cap[h]     = bytes;
        }
        b200conv_sp_frame_t *frames = reinterpret_cast<b200conv_sp_frame_t *>(s->h_tab[h]);
        SpFnInst *insts     = reinterpret_cast<SpFnInst *>(s->h_tab[h] + fn_at);
        size_t f            = 0;
        for (size_t j = 0; j < B; ++j)
        {
            insts[j]            = SpFnInst{ fi[j], uint32_t(f) };
            for (size_t p = (off[j] >= F) ? 0 : F - off[j]; p < len; p += F)
                frames[f++]         = b200conv_sp_frame_t{ fi[j], uint32_t(base + s0 + p) };
            off[j]              = sp_advance(off[j], len, F);
        }

        CU(sp_grow_async(reinterpret_cast<void **>(&s->d_tab), &s->tab_cap, bytes, st));
        CU(sp_grow_async(reinterpret_cast<void **>(&s->d_spectra), &s->spectra_cap,
                         std::max<size_t>(nf, 1) * N * sizeof(float2), st));
        CU(cudaMemcpyAsync(s->d_tab, s->h_tab[h], bytes, cudaMemcpyHostToDevice, st));
        CU(cudaEventRecord(s->ev_tab[h], st));
        s->tab_used[h]      = true;
        s->tab_cur          = h ^ 1;

        SpArgs a            = call;
        a.src              += s0;
        a.dst              += s0;
        a.count             = uint32_t(len);
        a.spectra           = s->d_spectra;
        a.fn                = reinterpret_cast<const SpFnInst *>(s->d_tab + fn_at);
        a.n_fn              = uint32_t(B);
        const uint32_t g    = uint32_t(std::min<size_t>(B, grid));
        CU(launch_sp(a, SP_K_FWD, s->rank, g, st));
        if (nf > 0)
        {
            s->in_fn            = true;
            s->fn(s->fn_user, reinterpret_cast<float *>(s->d_spectra), reinterpret_cast<const b200conv_sp_frame_t *>(s->d_tab),
                  frames, nf, s->rank, st);
            s->in_fn            = false;
        }
        CU(launch_sp(a, SP_K_INV, s->rank, g, st));
        s0                 += len;
    }
    return B200CONV_OK;
}

/* `base`: position of the call's first sample in the caller's process call (process_planar stages) */
static int sp_process_device_impl(b200conv_sp_t *s, float *dst, size_t dst_stride, const float *src, size_t src_stride,
                                  size_t count, void *stream, size_t base)
{
    if (s == nullptr)
        return fail(B200CONV_ERR_ARG, "b200conv_sp_process_device: NULL handle");
    SP_NOT_IN_FN(s, "b200conv_sp_process_device");
    if (count == 0)
        return B200CONV_OK;
    if ((dst == nullptr) || (src == nullptr) || (count >= (size_t(1) << 32)) ||
        ((s->n > 1) && ((src_stride < count) || (dst_stride < count))))
        return fail(B200CONV_ERR_ARG, "b200conv_sp_process_device: bad buffers");
    ENTER_DEVICE(s);
    cudaStream_t st = (stream != nullptr) ? cudaStream_t(stream) : s->stream;
    TRY(sp_commit(s, st));

    SpArgs a;
    memset(&a, 0, sizeof(a));
    a.tw            = s->tw[s->rank + 1];
    a.wnd           = s->d_wnd;
    a.src           = src;
    a.dst           = dst;
    a.stride_src    = src_stride;
    a.stride_dst    = dst_stride;
    a.inbuf         = s->d_in;
    a.outbuf        = s->d_out;
    a.table         = s->d_table;
    a.bound         = s->d_bound;
    a.off           = s->d_off;
    a.n_inst        = uint32_t(s->n);
    a.count         = uint32_t(count);
    /* one CTA per instance, as many resident CTAs as the device holds */
    uint32_t grid   = uint32_t((s->n < size_t(8 * s->sm_count)) ? s->n : size_t(8 * s->sm_count));
    /* k_sp walks every instance but the function-bound ones, which are walked in sub-calls after it */
    std::vector<uint32_t> fi;
    for (size_t i = 0; i < s->n; ++i)
        if (s->bound[i] == SP_FUNCTION)
            fi.push_back(uint32_t(i));
    if (fi.size() < s->n)
        CU(launch_sp(a, SP_K_SP, s->rank, grid, st));
    if (!fi.empty())
        TRY(sp_run_function(s, a, fi, count, base, grid, st));

    /* the host mirror of nOffset (remaining()), same arithmetic as the kernel's loop (:154-198) */
    const uint32_t F = uint32_t(1) << (s->rank - 1);
    for (size_t i = 0; i < s->n; ++i)
        s->h_off[i]     = sp_advance(s->h_off[i], count, F);
    return B200CONV_OK;
}

extern "C" int b200conv_sp_process_device(b200conv_sp_t *s, float *dst, size_t dst_stride, const float *src,
                                          size_t src_stride, size_t count, void *stream)
{
    try { return sp_process_device_impl(s, dst, dst_stride, src, src_stride, count, stream, 0); }
    catch (const std::bad_alloc &) { return fail(B200CONV_ERR_NOMEM, "out of host memory"); }
}

/* Host matrix [instances][stride] floats; synchronous (the reference's process() is). */
static int sp_process_planar_impl(b200conv_sp_t *s, float *dst, const float *src, size_t stride, size_t count)
{
    if (s == nullptr)
        return fail(B200CONV_ERR_ARG, "b200conv_sp_process_planar: NULL handle");
    SP_NOT_IN_FN(s, "b200conv_sp_process_planar");
    if (count == 0)
        return B200CONV_OK;
    if ((dst == nullptr) || (src == nullptr) || (stride < count))
        return fail(B200CONV_ERR_ARG, "b200conv_sp_process_planar: bad buffers");
    ENTER_DEVICE(s);
    size_t cap = (size_t(1) << 24) / s->n;
    if (cap > (size_t(1) << 20))    cap = size_t(1) << 20;
    if (cap < 1)                    cap = 1;
    size_t n_fn = 0;
    for (size_t i = 0; i < s->n; ++i)
        n_fn           += (s->bound[i] == SP_FUNCTION);
    if (n_fn > 0)
    {
        /* whole sub-calls of the spectral function per staged chunk where they fit */
        const size_t L  = sp_fn_span(s->rank, n_fn);
        if (L <= cap)
            cap             = cap / L * L;
    }
    for (size_t done = 0; done < count; )
    {
        const size_t c = (count - done < cap) ? count - done : cap;
        if (s->n * c > s->stage_floats)
        {
            CU(cudaStreamSynchronize(s->stream));
            if (s->sd_in)   cudaFree(s->sd_in);
            if (s->sd_out)  cudaFree(s->sd_out);
            s->sd_in = s->sd_out = nullptr;
            s->stage_floats = 0;
            CU(cudaMalloc(&s->sd_in, s->n * c * sizeof(float)));
            CU(cudaMalloc(&s->sd_out, s->n * c * sizeof(float)));
            s->stage_floats = s->n * c;
        }
        CU(cudaMemcpy2DAsync(s->sd_in, c * sizeof(float), src + done, stride * sizeof(float), c * sizeof(float), s->n,
                             cudaMemcpyHostToDevice, s->stream));
        TRY(sp_process_device_impl(s, s->sd_out, c, s->sd_in, c, c, s->stream, done));
        CU(cudaMemcpy2DAsync(dst + done, stride * sizeof(float), s->sd_out, c * sizeof(float), c * sizeof(float), s->n,
                             cudaMemcpyDeviceToHost, s->stream));
        CU(cudaStreamSynchronize(s->stream));
        done += c;
    }
    return B200CONV_OK;
}

extern "C" int b200conv_sp_process_planar(b200conv_sp_t *s, float *dst, const float *src, size_t stride, size_t count)
{
    try { return sp_process_planar_impl(s, dst, src, stride, count); }
    catch (const std::bad_alloc &) { return fail(B200CONV_ERR_NOMEM, "out of host memory"); }
}

extern "C" int b200conv_sp_reset(b200conv_sp_t *s)
{
    if (s == nullptr)
        return fail(B200CONV_ERR_ARG, "b200conv_sp_reset: NULL handle");
    SP_NOT_IN_FN(s, "b200conv_sp_reset");
    ENTER_DEVICE(s);
    const size_t N = size_t(1) << s->rank;
    for (size_t i = 0; i < s->n; ++i)
    {
        if (s->dirty[i])                            /* update_settings() will clear the buffers (:249-250) */
            continue;
        CU(cudaMemsetAsync(s->d_in + i * N, 0, N * sizeof(float), s->stream));      /* :256: pOutBuf, 2 N floats */
        CU(cudaMemsetAsync(s->d_out + i * N, 0, N * sizeof(float), s->stream));
    }
    return B200CONV_OK;
}

extern "C" int b200conv_sp_sync(b200conv_sp_t *s)
{
    if (s == nullptr)
        return fail(B200CONV_ERR_ARG, "b200conv_sp_sync: NULL handle");
    SP_NOT_IN_FN(s, "b200conv_sp_sync");
    ENTER_DEVICE(s);
    CU(cudaStreamSynchronize(s->stream));
    return B200CONV_OK;
}

extern "C" void *b200conv_sp_stream(b200conv_sp_t *s)              { return (s != nullptr) ? (void *)s->stream : nullptr; }
extern "C" size_t b200conv_sp_rank(const b200conv_sp_t *s)          { return (s != nullptr) ? s->rank : 0; }
extern "C" size_t b200conv_sp_latency(const b200conv_sp_t *s)       { return (s != nullptr) ? (size_t(1) << s->rank) : 0; }
extern "C" size_t b200conv_sp_instances(const b200conv_sp_t *s)     { return (s != nullptr) ? s->n : 0; }

/* SpectralProcessor::remaining (:241-245) */
extern "C" size_t b200conv_sp_remaining(const b200conv_sp_t *s, size_t idx)
{
    if ((s == nullptr) || (idx >= s->n))
        return 0;
    const size_t F = size_t(1) << (s->rank - 1);
    return (s->h_off[idx] <= F) ? F - s->h_off[idx] : 0;
}

#endif /* B200CONV_SPECTRAL_HOST_CUH_ */

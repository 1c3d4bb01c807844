/*
 * spectral.cuh -- lsp::dspu::SpectralProcessor, batched over many instances (scope-table row f4;
 * included by engine.cu).
 *
 * Reference: src/main/util/SpectralProcessor.cpp:147-199.  An STFT with a sine window before and
 * after the spectral operation (sin^2 + cos^2 = 1 at 50 % overlap): every N / 2 input samples
 * (N = 2^rank) the reference windows the last N samples, transforms them, hands the packed complex
 * spectrum to a callback, transforms back, windows again and overlap-adds into an output buffer
 * that is read N / 2 samples per frame -- N samples of latency (:SpectralProcessor.h latency()),
 * the first transform after N / 2 - size_t(N * (phase * 0.5f)) samples (:114-125).
 *
 * Here: ONE launch per process call for the whole batch (k_sp).  A CTA owns one instance and walks
 * the call exactly like the reference's loop (:154-198): sample exchange up to the next frame
 * boundary, transform, and so on -- instances with different phases need no host-side
 * scheduling.  Per instance the spectral operation is one of:
 *     none        reference: pFunc == NULL (:174-175), the frame is only windowed twice;
 *     table       spectrum[k] *= H[k] with a per-instance complex table (a real gain per bin is
 *                 the special case Im H = 0).  For ANY table of N bins the reference's result is
 *                 Re(IFFT(X H)); since the input is real that equals the inverse transform of
 *                 X[k] * (H[k] + conj(H[N-k])) / 2 over the N / 2 + 1 unique bins -- the table is
 *                 folded that way at bind time, so the device works on half spectra only;
 *     function    the caller's own device work on the full spectra (pFunc bound).  Within one call
 *                 every frame's input spectrum depends on the input only, so the call is split in
 *                 three stream-ordered steps: k_sp_fwd transforms every frame of the function-bound
 *                 instances into a slot of a spectra buffer, the host hands that buffer to the
 *                 caller's function, k_sp_inv folds each slot to its Hermitian part (what the
 *                 reference's Re(IFFT(X)) keeps), transforms back and overlap-adds.  k_sp skips
 *                 these instances.
 * A real N-point transform is one N / 2-point complex transform of z[m] = x[2m] + i x[2m+1]
 * (fft_smem at rank + 1 with ONE resident sequence) and a split / merge pass.
 */
#ifndef B200CONV_SPECTRAL_CUH_
#define B200CONV_SPECTRAL_CUH_

enum : uint8_t { SP_UNBOUND = 0, SP_TABLE = 1, SP_FUNCTION = 2 };  /* SpArgs::bound */

struct SpFnInst
{
    uint32_t        inst;           /* a function-bound instance                                    */
    uint32_t        first;          /* slot of its first frame of the call in SpArgs::spectra       */
};

struct SpArgs
{
    const float2   *tw;             /* twiddle table of transform rank `rank + 1` (FftCfg<rank + 1>)   */
    const float    *wnd;            /* [N] sine window, computed like the reference's (windows.cpp:238) */
    const float    *src;            /* [instances][stride_src]                                      */
    float          *dst;            /* [instances][stride_dst]                                      */
    uint64_t        stride_src, stride_dst;
    float          *inbuf;          /* [instances][N]  pInBuf  (SpectralProcessor.cpp:117)           */
    float          *outbuf;         /* [instances][N]  pOutBuf (:116)                                */
    const float2   *table;          /* [instances][N/2 + 1] folded tables, or NULL                   */
    const uint8_t  *bound;          /* [instances] SP_UNBOUND / SP_TABLE / SP_FUNCTION               */
    uint32_t       *off;            /* [instances] nOffset                                           */
    uint32_t        n_inst;
    uint32_t        count;          /* samples of this call                                          */
    /* k_sp_fwd / k_sp_inv only */
    float2         *spectra;        /* [frames][N] packed complex bins, one slot per frame           */
    const SpFnInst *fn;             /* [n_fn] function-bound instances, ascending                    */
    uint32_t        n_fn;
};

/* RANKP = rank + 1: FftCfg<RANKP, 0, 1> is ONE sequence of P = 2^(rank - 1) = N / 2 complex points. */
template <int RANKP>
struct SpCfg
{
    using C = FftCfg<RANKP, 0, 1>;
    static constexpr int  P     = C::P;             /* complex points = N / 2 = frame size          */
    static constexpr int  N     = 2 * P;
    static constexpr bool PP    = (RANKP <= 13);    /* second work buffer (<= 32 KiB each)            */
    static constexpr bool TWS   = (RANKP <= 12);    /* whole twiddle table in shared memory           */
    static constexpr int  TWN   = TWS ? C::TW_TOTAL : C::TWC_N;
    static constexpr size_t SMEM = (size_t(P) * (PP ? 2 : 1) + TWN) * sizeof(float2);
};

/* Stages the twiddles of the CTA; returns w_N^k = exp(-2 pi i k / N), k < N / 2: the "pre" third of
 * the rank + 1 table (w_M'^m, M' = N). */
template <int RANKP>
__device__ __forceinline__ const float2 *sp_stage_twiddles(float2 *tws, const float2 *tw, int tid)
{
    using S = SpCfg<RANKP>;
    using C = typename S::C;
    if (S::TWS)
        for (int i = tid; i < C::TW_TOTAL; i += C::T)
            tws[i]              = tw[i];
    else
        stage_compact_twiddles<C>(tws, tw, tid);
    __syncthreads();
    return (S::TWS ? tws : tw) + C::TW_PRE;
}

/* :163-164 window, :165 forward transform (as N / 2 complex points); returns the buffer holding Z */
template <int RANKP>
__device__ __forceinline__ float2 *sp_window_forward(const float *inb, const float *wnd, float2 *A, float2 *B,
                                                     const float2 *tws, int tid)
{
    using S = SpCfg<RANKP>;
    for (int m = tid; m < S::P; m += S::C::T)
    {
        const float2 x  = reinterpret_cast<const float2 *>(inb)[m];
        const float2 w  = reinterpret_cast<const float2 *>(wnd)[m];
        A[m]            = make_float2(x.x * w.x, x.y * w.y);
    }
    __syncthreads();
    return fft_smem<RANKP, false, S::PP, 0, true, true, 1, !S::TWS>(A, B, tws, tid);
}

/* split: X[k] and X[P - k] of the real N-point transform from the half-size transform Z, 1 <= k <= P / 2:
 * E = (Zk + conj(Zm)) / 2, O = -i (Zk - conj(Zm)) / 2, X[k] = E + w O, X[P-k] = conj(E) - conj(w O) */
__device__ __forceinline__ void sp_split(float2 zk, float2 zm, float2 w, float2 &Xk, float2 &Xm)
{
    const float2 E  = make_float2(0.5f * (zk.x + zm.x), 0.5f * (zk.y - zm.y));
    const float2 O  = make_float2(0.5f * (zk.y + zm.y), -0.5f * (zk.x - zm.x));
    const float2 wO = cmul(w, O);
    Xk              = make_float2(E.x + wO.x, E.y + wO.y);
    Xm              = make_float2(E.x - wO.x, -E.y + wO.y);
}

/* merge, the inverse of sp_split: E' = (Xk + conj(Xm)) / 2, w O' = (Xk - conj(Xm)) / 2,
 * Z'[k] = E' + i O', Z'[P-k] = conj(E') + i conj(O') */
__device__ __forceinline__ void sp_merge(float2 Xk, float2 Xm, float2 w, float2 &Dk, float2 &Dm)
{
    const float2 E2 = make_float2(0.5f * (Xk.x + Xm.x), 0.5f * (Xk.y - Xm.y));
    const float2 O2 = cmulc(make_float2(0.5f * (Xk.x - Xm.x), 0.5f * (Xk.y + Xm.y)), w);
    Dk              = make_float2(E2.x - O2.y, E2.y + O2.x);
    Dm              = make_float2(E2.x + O2.y, O2.x - E2.y);
}

/* :167 reverse transform of D (1 / P: the half-size transform carries the whole scale); :172-174
 * shift the output buffer, clear its tail, add the frame windowed again */
template <int RANKP>
__device__ __forceinline__ void sp_inverse_ola(float2 *D, float2 *E, float2 *A, const float2 *tws, const float *wnd,
                                               float *outb, int tid)
{
    using S = SpCfg<RANKP>;
    constexpr int P = S::P, T = S::C::T;
    float2 *Y           = fft_smem<RANKP, true, S::PP, 0, true, true, 1, !S::TWS>(D, E, tws, tid);
    const float scale   = 1.0f / float(P);
    for (int m = tid; m < P; m += T)
    {
        const float2 y  = Y[m];
        const float2 w  = reinterpret_cast<const float2 *>(wnd)[m];
        float2 o        = (2 * m < P) ? reinterpret_cast<const float2 *>(outb)[m + P / 2] : make_float2(0.0f, 0.0f);
        o.x            += y.x * scale * w.x;
        o.y            += y.y * scale * w.y;
        A[m]            = o;            /* staged: outb[m] still feeds outb[m - P / 2] */
    }
    __syncthreads();
    for (int m = tid; m < P; m += T)
        reinterpret_cast<float2 *>(outb)[m] = A[m];
}

template <int RANKP>
__global__ void __launch_bounds__(FftCfg<RANKP, 0, 1>::T)
k_sp(const SpArgs a)
{
    using S = SpCfg<RANKP>;
    using C = typename S::C;
    constexpr int P = S::P, N = S::N, T = C::T;
    extern __shared__ float2 sp_sm[];
    float2 *A               = sp_sm;
    float2 *B               = S::PP ? sp_sm + P : nullptr;
    float2 *tws             = sp_sm + P * (S::PP ? 2 : 1);
    const int tid           = threadIdx.x;

    if (S::TWS)
        for (int i = tid; i < C::TW_TOTAL; i += T)
            tws[i]              = a.tw[i];
    else
        stage_compact_twiddles<C>(tws, a.tw, tid);
    __syncthreads();
    /* w_N^k = exp(-2 pi i k / N), k < N / 2, is the "pre" third of the rank + 1 table (w_M'^m, M' = N) */
    const float2 *wN        = (S::TWS ? tws : a.tw) + C::TW_PRE;

    for (uint32_t inst = blockIdx.x; inst < a.n_inst; inst += gridDim.x)
    {
        float *inb              = a.inbuf + uint64_t(inst) * N;
        float *outb             = a.outbuf + uint64_t(inst) * N;
        const float *src        = a.src + uint64_t(inst) * a.stride_src;
        float *dst              = a.dst + uint64_t(inst) * a.stride_dst;
        if (a.bound[inst] == SP_FUNCTION)
            continue;
        const bool bound        = (a.table != nullptr) && (a.bound[inst] == SP_TABLE);
        const float2 *H         = bound ? a.table + uint64_t(inst) * (P + 1) : nullptr;
        uint32_t off            = a.off[inst];
        uint32_t pos            = 0;

        while (pos < a.count)                                       /* SpectralProcessor.cpp:154 */
        {
            if (off >= uint32_t(P))                                 /* :157 : a frame boundary */
            {
                if (bound)
                {
                    /* :163-164 window, :165 forward transform (as N / 2 complex points) */
                    for (int m = tid; m < P; m += T)
                    {
                        const float2 x  = reinterpret_cast<const float2 *>(inb)[m];
                        const float2 w  = reinterpret_cast<const float2 *>(a.wnd)[m];
                        A[m]            = make_float2(x.x * w.x, x.y * w.y);
                    }
                    __syncthreads();
                    float2 *Z           = fft_smem<RANKP, false, S::PP, 0, true, true, 1, !S::TWS>(A, B, tws, tid);
                    float2 *D           = S::PP ? ((Z == A) ? B : A) : Z;
                    /* split -> X[k], :166 the spectral operation X[k] *= H[k], merge -> Z'[k];
                     * pairs (k, P - k) in registers, in place when there is one work buffer.  The
                     * algebra of sp_split / sp_merge, kept inline here: through the helpers ptxas
                     * allocates this kernel differently and spills at rank 11 */
                    for (int k = tid; k <= P / 2; k += T)
                    {
                        const int km    = P - k;
                        if (k == 0)
                        {
                            const float2 z0 = Z[0];
                            const float x0  = (z0.x + z0.y) * H[0].x;               /* DC: real        */
                            const float xn  = (z0.x - z0.y) * H[P].x;               /* Nyquist: real   */
                            D[0]            = make_float2(0.5f * (x0 + xn), 0.5f * (x0 - xn));
                            continue;
                        }
                        const float2 zk = Z[k], zm = Z[km];
                        const float2 w  = wN[k];
                        /* E = (Zk + conj(Zm)) / 2, O = -i (Zk - conj(Zm)) / 2, X[k] = E + w O, X[P-k] = conj(E) - conj(w O) */
                        const float2 E  = make_float2(0.5f * (zk.x + zm.x), 0.5f * (zk.y - zm.y));
                        const float2 O  = make_float2(0.5f * (zk.y + zm.y), -0.5f * (zk.x - zm.x));
                        const float2 wO = cmul(w, O);
                        float2 Xk       = cmul(make_float2(E.x + wO.x, E.y + wO.y), H[k]);
                        float2 Xm       = cmul(make_float2(E.x - wO.x, -E.y + wO.y), H[km]);
                        /* E' = (Xk + conj(Xm)) / 2, w O' = (Xk - conj(Xm)) / 2, Z'[k] = E' + i O', Z'[P-k] = conj(E') + i conj(O') */
                        const float2 E2 = make_float2(0.5f * (Xk.x + Xm.x), 0.5f * (Xk.y - Xm.y));
                        const float2 O2 = cmulc(make_float2(0.5f * (Xk.x - Xm.x), 0.5f * (Xk.y + Xm.y)), w);
                        D[k]            = make_float2(E2.x - O2.y, E2.y + O2.x);
                        if (km != k)
                            D[km]           = make_float2(E2.x + O2.y, O2.x - E2.y);
                    }
                    __syncthreads();
                    /* :167 reverse transform (1 / P: the half-size transform carries the whole scale) */
                    float2 *Y           = fft_smem<RANKP, true, S::PP, 0, true, true, 1, !S::TWS>(D, S::PP ? Z : nullptr, tws, tid);
                    const float scale   = 1.0f / float(P);
                    /* :172-174 shift the output buffer, clear its tail, add the frame windowed again */
                    for (int m = tid; m < P; m += T)
                    {
                        const float2 y  = Y[m];
                        const float2 w  = reinterpret_cast<const float2 *>(a.wnd)[m];
                        float2 o        = (2 * m < P) ? reinterpret_cast<const float2 *>(outb)[m + P / 2] : make_float2(0.0f, 0.0f);
                        o.x            += y.x * scale * w.x;
                        o.y            += y.y * scale * w.y;
                        A[m]            = o;            /* staged: outb[m] still feeds outb[m - P / 2] */
                    }
                    __syncthreads();
                    for (int m = tid; m < P; m += T)
                        reinterpret_cast<float2 *>(outb)[m] = A[m];
                }
                else
                {
                    /* :174-175 no operation bound: the frame is only windowed, twice; :172-174 shift,
                     * clear, add -- element i and i + P belong to the same thread */
                    for (int i = tid; i < P; i += T)
                    {
                        const float w0  = a.wnd[i], w1 = a.wnd[i + P];
                        const float lo  = outb[i + P] + inb[i] * w0 * w0;
                        const float hi  = inb[i + P] * w1 * w1;
                        outb[i]         = lo;
                        outb[i + P]     = hi;
                    }
                }
                __syncthreads();
                /* :177 shift the input buffer */
                for (int i = tid; i < P; i += T)
                    inb[i]              = inb[i + P];
                off                 = 0;
                __syncthreads();
            }

            /* :184-189 exchange samples up to the next frame boundary */
            const uint32_t n    = min(uint32_t(P) - off, a.count - pos);
            for (uint32_t i = tid; i < n; i += T)
            {
                const float v       = src[pos + i];
                dst[pos + i]        = outb[off + i];
                inb[P + off + i]    = v;
            }
            off                += n;
            pos                += n;
            __syncthreads();
        }
        if (tid == 0)
            a.off[inst]         = off;
    }
}

/* First step of a call for the function-bound instances: the input half of k_sp's walk.  At every
 * frame boundary the windowed frame is transformed and its N bins go to the frame's slot -- X[k]
 * for k <= N / 2 and conj(X[k]) at N - k, the reference's packed layout.  The input buffer is
 * shifted as in k_sp; nOffset is read, not written (k_sp_inv walks the same call after it). */
template <int RANKP>
__global__ void __launch_bounds__(FftCfg<RANKP, 0, 1>::T)
k_sp_fwd(const SpArgs a)
{
    using S = SpCfg<RANKP>;
    using C = typename S::C;
    constexpr int P = S::P, N = S::N, T = C::T;
    extern __shared__ float2 sp_sm[];
    float2 *A               = sp_sm;
    float2 *B               = S::PP ? sp_sm + P : nullptr;
    float2 *tws             = sp_sm + P * (S::PP ? 2 : 1);
    const int tid           = threadIdx.x;
    const float2 *wN        = sp_stage_twiddles<RANKP>(tws, a.tw, tid);

    for (uint32_t j = blockIdx.x; j < a.n_fn; j += gridDim.x)
    {
        const uint32_t inst     = a.fn[j].inst;
        uint32_t slot           = a.fn[j].first;
        float *inb              = a.inbuf + uint64_t(inst) * N;
        const float *src        = a.src + uint64_t(inst) * a.stride_src;
        uint32_t off            = a.off[inst];
        uint32_t pos            = 0;

        while (pos < a.count)
        {
            if (off >= uint32_t(P))
            {
                const float2 *Z     = sp_window_forward<RANKP>(inb, a.wnd, A, B, tws, tid);
                float2 *X           = a.spectra + uint64_t(slot++) * N;
                for (int k = tid; k <= P / 2; k += T)
                {
                    const int km    = P - k;
                    if (k == 0)
                    {
                        const float2 z0 = Z[0];
                        X[0]            = make_float2(z0.x + z0.y, 0.0f);           /* DC      */
                        X[P]            = make_float2(z0.x - z0.y, 0.0f);           /* Nyquist */
                        continue;
                    }
                    float2 Xk, Xm;
                    sp_split(Z[k], Z[km], wN[k], Xk, Xm);
                    X[k]            = Xk;
                    X[N - k]        = make_float2(Xk.x, -Xk.y);
                    if (km != k)
                    {
                        X[km]           = Xm;
                        X[N - km]       = make_float2(Xm.x, -Xm.y);
                    }
                }
                /* the window read inb before the transform's first barrier */
                for (int i = tid; i < P; i += T)
                    inb[i]              = inb[i + P];
                off                 = 0;
                __syncthreads();
            }

            const uint32_t n    = min(uint32_t(P) - off, a.count - pos);
            for (uint32_t i = tid; i < n; i += T)
                inb[P + off + i]    = src[pos + i];
            off                += n;
            pos                += n;
            __syncthreads();
        }
    }
}

/* Last step of a call for the function-bound instances: the output half of k_sp's walk.  At every
 * frame boundary the slot Y of the frame is folded to its Hermitian part (Y[k] + conj(Y[N - k])) / 2
 * -- the reference keeps Re(IFFT(Y)) only -- and merged, transformed back and overlap-added;
 * samples leave from the output buffer; nOffset is written back. */
template <int RANKP>
__global__ void __launch_bounds__(FftCfg<RANKP, 0, 1>::T)
k_sp_inv(const SpArgs a)
{
    using S = SpCfg<RANKP>;
    using C = typename S::C;
    constexpr int P = S::P, N = S::N, T = C::T;
    extern __shared__ float2 sp_sm[];
    float2 *A               = sp_sm;
    float2 *B               = S::PP ? sp_sm + P : nullptr;
    float2 *tws             = sp_sm + P * (S::PP ? 2 : 1);
    const int tid           = threadIdx.x;
    const float2 *wN        = sp_stage_twiddles<RANKP>(tws, a.tw, tid);

    for (uint32_t j = blockIdx.x; j < a.n_fn; j += gridDim.x)
    {
        const uint32_t inst     = a.fn[j].inst;
        uint32_t slot           = a.fn[j].first;
        float *outb             = a.outbuf + uint64_t(inst) * N;
        float *dst              = a.dst + uint64_t(inst) * a.stride_dst;
        uint32_t off            = a.off[inst];
        uint32_t pos            = 0;

        while (pos < a.count)
        {
            if (off >= uint32_t(P))
            {
                const float2 *Y     = a.spectra + uint64_t(slot++) * N;
                for (int k = tid; k <= P / 2; k += T)
                {
                    const int km    = P - k;
                    if (k == 0)
                    {
                        const float x0  = Y[0].x, xn = Y[P].x;                      /* Hermitian parts of DC, Nyquist */
                        A[0]            = make_float2(0.5f * (x0 + xn), 0.5f * (x0 - xn));
                        continue;
                    }
                    const float2 yk = Y[k], ykc = Y[N - k], ym = Y[km], ymc = Y[N - km];
                    const float2 Xk = make_float2(0.5f * (yk.x + ykc.x), 0.5f * (yk.y - ykc.y));
                    const float2 Xm = make_float2(0.5f * (ym.x + ymc.x), 0.5f * (ym.y - ymc.y));
                    float2 Dk, Dm;
                    sp_merge(Xk, Xm, wN[k], Dk, Dm);
                    A[k]            = Dk;
                    if (km != k)
                        A[km]           = Dm;
                }
                __syncthreads();
                sp_inverse_ola<RANKP>(A, B, A, tws, a.wnd, outb, tid);
                off                 = 0;
                __syncthreads();
            }

            const uint32_t n    = min(uint32_t(P) - off, a.count - pos);
            for (uint32_t i = tid; i < n; i += T)
                dst[pos + i]        = outb[off + i];
            off                += n;
            pos                += n;
            __syncthreads();
        }
        if (tid == 0)
            a.off[inst]         = off;
    }
}

#endif /* B200CONV_SPECTRAL_CUH_ */

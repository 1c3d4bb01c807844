/*
 * matrix.cuh -- sm_100a device code of the matrix convolver (b200conv_mx_*; included by engine.cu
 * after kernels.cuh, host side in matrix_host.cuh).
 *
 * I inputs, O outputs, a list of routes (input i, output o, impulse response h):
 *     y_o = sum over the routes r into o of  h_r (*) x_in(r)
 * The arithmetic plan is the convolver's (uniform partitions of F, folded overlap, a frequency-domain
 * delay line); what changes is what is shared.  Each INPUT has one spectrum ring, filled by k_fwd;
 * each OUTPUT has one inverse transform, k_inv, which sums the partial rows of every route into it.
 * The only new kernel is the partition MAC below, which reads an input's ring rows ONCE for up to
 * MX_RG routes leaving that input.
 */
#ifndef B200CONV_MATRIX_CUH_
#define B200CONV_MATRIX_CUH_

namespace b200conv
{

/* Routes per k_mx_mac CTA.  Rank 11 (TB = M = 1024, QB = 1), two stages: a stage holds one ring row
 * and MX_RG IR rows, 8 KiB each, so 2 x 5 x 8 KiB = 80 KiB of shared memory per CTA and two CTAs per
 * SM; -Xptxas -v: 96 registers, no spills, under the 128 that __launch_bounds__(256, 2) allows.
 * MX_RG = 8 would read a fan-out input's ring half as often but leaves one 144 KiB CTA per SM, which
 * cannot keep enough bulk copies in flight to stream from HBM. */
constexpr int MX_RG     = 4;
constexpr int MX_STAGES = 2;        /* as k_mac: two stages of one partition row measured best */

struct MxUnit                       /* one group of routes leaving one input; device resident */
{
    const float2   *G[MX_RG];       /* [nq][M] folded IR spectra of each route                   */
    uint32_t        nq[MX_RG];      /* rows of G; 0 for the unused slots r >= nr                  */
    uint32_t        row[MX_RG];     /* partial row of split 0 within a frame: output * rows +
                                       (rank of the route among the routes into that output) * splits */
    uint32_t        input;
    uint32_t        nr;             /* routes in the group, 1 .. MX_RG */
    uint32_t        nq_max;         /* partitions the splits of the group divide */
    uint32_t        pad;
};

struct MxArgs                       /* by-value kernel argument */
{
    const MxUnit   *units;
    const float2   *ring;           /* [inputs][S][M]: frame t of input i in slot (-t) mod S      */
    float2         *ypart;          /* [frame of the launch][outputs][rows][M]                    */
    uint64_t        t_base;         /* frame index (since set_routes / clear) of the launch's frame 0 */
    uint32_t        S, rank, splits, rows, outputs;
    uint32_t        TB, QB, rg;     /* bins per CTA tile, partitions per stage, IR rows per stage */
};

/* grid = (units * splits, M / TB, frames).  A CTA streams the partitions [q0, q1) of its split for its
 * group: per stage one bulk copy of the input's ring rows (two around the ring's wrap) and one per
 * route of its G rows; a route shorter than the range skips its copies and FMAs for the partitions it
 * does not have (a test on the stage's partition index: uniform over the CTA). */
__global__ void __launch_bounds__(256, 2)
k_mx_mac(const MxArgs a)
{
    extern __shared__ __align__(128) unsigned char smraw[];

    /* the k_inv launched behind this one stages its twiddles now and waits for completion */
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

    const uint32_t M        = 1u << (a.rank - 1);
    const uint32_t TB       = a.TB, QB = a.QB, NS = MX_STAGES;
    const uint32_t T        = blockDim.x;
    const uint32_t tid      = threadIdx.x;
    const uint32_t ui       = blockIdx.x / a.splits;
    const uint32_t split    = blockIdx.x % a.splits;
    const uint32_t tile     = blockIdx.y;
    const uint32_t z        = blockIdx.z;
    const MxUnit &u         = a.units[ui];
    const uint32_t nr       = u.nr;

    uint32_t nq[MX_RG];
    const float2 *Gt[MX_RG];
    #pragma unroll
    for (int r = 0; r < MX_RG; ++r)
    {
        nq[r]               = (uint32_t(r) < nr) ? u.nq[r] : 0u;
        Gt[r]               = (uint32_t(r) < nr) ? u.G[r] + uint64_t(tile) * TB : nullptr;
    }

    const uint32_t stage_elems = QB * TB;                           /* float2 per operand per stage */
    float2 *sX              = reinterpret_cast<float2 *>(smraw);    /* [NS][stage_elems]     */
    float2 *sG              = sX + size_t(NS) * stage_elems;        /* [NS][rg][stage_elems] */
    uint64_t *full          = reinterpret_cast<uint64_t *>(sG + size_t(NS) * a.rg * stage_elems);

    uint32_t q0, q1;
    chunk_range(u.nq_max, split, a.splits, 0, q0, q1);
    const uint32_t n_iter   = (q1 - q0 + QB - 1) / QB;

    const uint64_t t        = a.t_base + z;
    const uint32_t tm       = uint32_t(t % a.S);
    const uint32_t slot0    = (tm == 0) ? 0 : a.S - tm;
    const float2 *Xt        = a.ring + uint64_t(u.input) * a.S * M + uint64_t(tile) * TB;
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

    /* One frame per launch: partition 0 needs the spectrum the k_fwd right before this launch is
     * writing, so the CTAs that own it visit their stages in the order 1, 2, ..., n_iter - 1, 0 and
     * wait for that launch only in front of the last one (as k_mac with STEP_AFTER_FWD).  Every other
     * ring row and every IR row is final when this launch starts.  Several frames: wait first. */
    const uint32_t late     = ((gridDim.z == 1) && (q0 == 0) && (n_iter > 0)) ? 1u : 0u;
    const uint32_t slot_q0  = uint32_t((uint64_t(slot0) + q0) % a.S);
    uint32_t f_it = 0, f_s = 0, f_q = q0 + late * QB;
    uint32_t f_slot         = slot_q0 + late * QB;
    if (f_slot >= a.S)      f_slot -= a.S;
    auto issue_next = [&]()
    {
        if (late && (f_it == n_iter - 1))
        {
            asm volatile("griddepcontrol.wait;" ::: "memory");
            asm volatile("fence.proxy.async;" ::: "memory");
            f_q             = q0;
            f_slot          = slot_q0;
        }
        const uint32_t rows = min(QB, q1 - f_q);
        uint32_t rr[MX_RG];
        uint32_t total  = rows;
        #pragma unroll
        for (int r = 0; r < MX_RG; ++r)
        {
            rr[r]           = (f_q < nq[r]) ? min(rows, nq[r] - f_q) : 0u;
            total          += rr[r];
        }
        mbar_expect_tx(&full[f_s], total * row_bytes);
        float2 *x       = sX + size_t(f_s) * stage_elems;
        /* TB < M only at ranks >= 12, where QB == 1: a stage is one row either way */
        const uint32_t n1 = min(rows, a.S - f_slot);
        bulk_g2s(x, Xt + uint64_t(f_slot) * M, n1 * row_bytes, &full[f_s], l2_stream);
        if (n1 < rows)
            bulk_g2s(x + size_t(n1) * TB, Xt, (rows - n1) * row_bytes, &full[f_s], l2_stream);
        #pragma unroll
        for (int r = 0; r < MX_RG; ++r)
            if (rr[r] > 0)
                bulk_g2s(sG + (size_t(f_s) * a.rg + r) * stage_elems, Gt[r] + uint64_t(f_q) * M, rr[r] * row_bytes,
                         &full[f_s], l2_stream);
        ++f_it;
        f_q            += QB;
        f_slot         += QB;
        if (f_slot >= a.S)  f_slot -= a.S;
        if (++f_s == NS)    f_s = 0;
    };

    if (tid == 0)
    {
        if ((gridDim.z > 1) && (n_iter > 0))
        {
            asm volatile("griddepcontrol.wait;" ::: "memory");
            asm volatile("fence.proxy.async;" ::: "memory");
        }
        while ((f_it < NS) && (f_it < n_iter))
            issue_next();
    }

    float4 acc[MX_RG][MAC_VPT];
    float dny[MX_RG];               /* per route: sum of Im*Im of the thread's first bin (Nyquist fix-up of bin 0) */
    #pragma unroll
    for (int r = 0; r < MX_RG; ++r)
    {
        dny[r]          = 0.0f;
        #pragma unroll
        for (int v = 0; v < MAC_VPT; ++v)
            acc[r][v]       = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    }

    uint32_t c_s = 0, c_par = 0, c_q = q0 + late * QB;
    for (uint32_t it = 0; it < n_iter; ++it)
    {
        if (late && (it == n_iter - 1))
            c_q             = q0;
        const uint32_t rows = min(QB, q1 - c_q);
        mbar_wait(&full[c_s], c_par);

        const float4 *x4 = reinterpret_cast<const float4 *>(sX + size_t(c_s) * stage_elems);
        const float4 *g4 = reinterpret_cast<const float4 *>(sG + size_t(c_s) * a.rg * stage_elems);
        for (uint32_t row = 0; row < rows; ++row)
        {
            float4 x[MAC_VPT];
            #pragma unroll
            for (int v = 0; v < MAC_VPT; ++v)
                x[v]            = x4[row * (TB / 2) + tid + v * T];
            #pragma unroll
            for (int r = 0; r < MX_RG; ++r)
            {
                if (c_q + row >= nq[r])
                    continue;
                #pragma unroll
                for (int v = 0; v < MAC_VPT; ++v)
                {
                    const float4 g  = g4[size_t(r) * (stage_elems / 2) + row * (TB / 2) + tid + v * T];
                    acc[r][v].x     = fmaf(g.x, x[v].x, acc[r][v].x);
                    acc[r][v].y     = fmaf(g.x, x[v].y, acc[r][v].y);
                    acc[r][v].z     = fmaf(g.z, x[v].z, acc[r][v].z);
                    acc[r][v].w     = fmaf(g.z, x[v].w, acc[r][v].w);
                    acc[r][v].x     = fmaf(-g.y, x[v].y, acc[r][v].x);
                    acc[r][v].y     = fmaf(g.y, x[v].x, acc[r][v].y);
                    acc[r][v].z     = fmaf(-g.w, x[v].w, acc[r][v].z);
                    acc[r][v].w     = fmaf(g.w, x[v].z, acc[r][v].w);
                    if (v == 0)
                        dny[r]          = fmaf(g.y, x[v].y, dny[r]);
                }
            }
        }
        c_q            += QB;
        if (++c_s == NS)    { c_s = 0; c_par ^= 1u; }

        __syncthreads();            /* everyone is done with that stage: refill it */
        if ((tid == 0) && (f_it < n_iter))
            issue_next();
    }

    /* bin 0 holds (DC, Nyquist): both real, multiplied separately.  The complex MAC above gave
     * x = sum(re*re - im*im), so re = x + sum(im*im), im = sum(im*im) -- for every route. */
    if ((tile == 0) && (tid == 0))
    {
        #pragma unroll
        for (int r = 0; r < MX_RG; ++r)
        {
            acc[r][0].x    += dny[r];
            acc[r][0].y     = dny[r];
        }
    }

    /* the rows are free: the k_inv that last read them completed before this launch's k_fwd started */
    float2 *yb      = a.ypart + uint64_t(z) * a.outputs * a.rows * M + uint64_t(tile) * TB;
    #pragma unroll
    for (int r = 0; r < MX_RG; ++r)
    {
        if (uint32_t(r) >= nr)
            continue;
        float4 *yp      = reinterpret_cast<float4 *>(yb + uint64_t(u.row[r] + split) * M);
        #pragma unroll
        for (int v = 0; v < MAC_VPT; ++v)
            yp[tid + v * T] = acc[r][v];
    }

    /* completion order: this launch completes after the k_fwd before it, so the k_inv behind it
     * writes the output only once every input block of the launch group has been read */
    if ((tid == 0) && (!late) && (gridDim.z == 1))
        asm volatile("griddepcontrol.wait;" ::: "memory");
    if ((tid == 0) && (n_iter == 0) && (gridDim.z > 1))
        asm volatile("griddepcontrol.wait;" ::: "memory");
}

/* ---- impulse-response replacement with a crossfade (b200conv_mx_set_irs) --------------------------
 * The ring holds input spectra only and no state crosses a block boundary, so by linearity
 *     y_o = IFFT(A + B_old) + w(n) * IFFT(B_delta),   B_delta = sum_q (G_new - G_old)_q X_{t-q}
 * where A sums the unchanged routes into o and B_old the old IRs of the changed ones.  The delta terms
 * are extra "delta routes" into extra "delta outputs" of k_mx_mac and k_inv; the two kernels below
 * ingest the new IRs and blend the delta outputs into the real ones. */

struct FoldDeltaDesc                /* one changed route */
{
    float2         *G;              /* [bins + 1][M] folded spectra of the new IR                  */
    float2         *D;              /* [nd][M] G_new - G_old, each zero-extended to nd rows; NULL:
                                       no fade, G_new only (nd = bins + 1)                           */
    const float2   *G_old;          /* [nq_old][M] the route's current folded spectra               */
    uint64_t        h_row;          /* first row of the route in the H slab                         */
    uint32_t        bins;           /* partitions of the new IR                                     */
    uint32_t        nq_old;
    uint32_t        nd;             /* max(bins + 1, nq_old)                                         */
    uint32_t        pad;
};

/* k_fold_many's fold of H into G_new, and G_new - G_old, in one pass */
__global__ void k_fold_delta(const FoldDeltaDesc *desc, uint32_t n, const float2 *H, uint32_t M)
{
    for (uint32_t i = blockIdx.z; i < n; i += gridDim.z)
    {
        const FoldDeltaDesc d = desc[i];
        const float2 *Hi    = H + d.h_row * M;
        for (uint32_t q = blockIdx.y; q < d.nd; q += gridDim.y)
        for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < M; k += gridDim.x * blockDim.x)
        {
            float2 g        = make_float2(0.0f, 0.0f);
            if (q <= d.bins)
            {
                float2 cur      = (q < d.bins) ? Hi[uint64_t(q) * M + k] : make_float2(0.0f, 0.0f);
                float2 prev     = (q > 0) ? Hi[uint64_t(q - 1) * M + k] : make_float2(0.0f, 0.0f);
                float sgn       = (k & 1) ? -1.0f : 1.0f;
                g               = make_float2(cur.x + sgn * prev.x, cur.y + sgn * prev.y);
                d.G[uint64_t(q) * M + k] = g;
            }
            if (d.D == nullptr)
                continue;
            const float2 o  = (q < d.nq_old) ? d.G_old[uint64_t(q) * M + k] : make_float2(0.0f, 0.0f);
            d.D[uint64_t(q) * M + k] = make_float2(g.x - o.x, g.y - o.y);
        }
    }
}

/* dst[omap[d]][z * F + n] += w(k) * delta[z][d][n] with k = k0 + z * F + n the sample index since the
 * fade began and w(k) = min(1, (k + 1) / fade): exact wherever the fade ends.  grid = (., deltas, frames);
 * launched after the k_inv that wrote both, so dst == src calls stay safe. */
__global__ void k_mx_blend(float *dst, uint64_t dst_stride, const float *delta, const uint32_t *omap,
                           uint32_t deltas, uint32_t F, uint64_t k0, uint64_t fade)
{
    const uint32_t di   = blockIdx.y, z = blockIdx.z;
    const float *dz     = delta + (uint64_t(z) * deltas + di) * F;
    float *y            = dst + uint64_t(omap[di]) * dst_stride + uint64_t(z) * F;
    for (uint32_t n = blockIdx.x * blockDim.x + threadIdx.x; n < F; n += gridDim.x * blockDim.x)
    {
        const uint64_t k    = k0 + uint64_t(z) * F + n;
        const float w       = (k + 1 >= fade) ? 1.0f : float(double(k + 1) / double(fade));
        y[n]                = fmaf(w, dz[n], y[n]);
    }
}

}   /* namespace b200conv */

#endif /* B200CONV_MATRIX_CUH_ */

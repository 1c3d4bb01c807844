/*
 * batch_fade.cuh -- the two kernels of a batch crossfade (b200conv_set_irs, DESIGN.md §4.8).
 *
 * While instances of a batch fade, each process call runs on one stream:
 *   k_fade_gather   the fading rows of src -> a compact matrix [slot][count] (before anything writes
 *                   dst: dst == src is allowed);
 *   the twin batch's call on that matrix: the fading instances with their NEW impulse responses
 *                   and a copy of their input history -> y_new [slot][count];
 *   the batch's own call, unchanged (the OLD impulse responses);
 *   k_fade_blend    dst[row] += w * (y_new - dst[row]).
 * Both kernels are plain launches: no programmatic serialisation, no early trigger.
 */
#ifndef B200CONV_BATCH_FADE_CUH_
#define B200CONV_BATCH_FADE_CUH_

namespace b200conv
{

/* one slot of the twin batch */
struct FadeRow
{
    int64_t     row;        /* the fading instance; < 0: free slot */
    uint64_t    start;      /* the batch's sample clock at set_irs */
    uint64_t    fade;       /* samples */
};

__global__ void k_fade_gather(float *out, const float *src, uint64_t src_stride, const FadeRow *rows,
                              uint32_t slots, uint64_t count)
{
    for (uint32_t s = blockIdx.y; s < slots; s += gridDim.y)
    {
        const int64_t row   = rows[s].row;
        if (row < 0)
            continue;
        const float *x      = src + uint64_t(row) * src_stride;
        float *y            = out + uint64_t(s) * count;
        for (uint64_t i = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < count; i += uint64_t(gridDim.x) * blockDim.x)
            y[i]                = x[i];
    }
}

/* dst[row][i] += w(k) * (y_new[slot][i] - dst[row][i]) with k = clock - start + i the sample index since
 * the fade began and w(k) = min(1, (k + 1) / fade); where w = 1 the new output is stored as it is, so
 * the samples after the fade are exactly the new IR's. */
__global__ void k_fade_blend(float *dst, uint64_t dst_stride, const float *y_new, const FadeRow *rows,
                             uint32_t slots, uint64_t count, uint64_t clock)
{
    for (uint32_t s = blockIdx.y; s < slots; s += gridDim.y)
    {
        const FadeRow r     = rows[s];
        if (r.row < 0)
            continue;
        const float *yn     = y_new + uint64_t(s) * count;
        float *y            = dst + uint64_t(r.row) * dst_stride;
        const uint64_t k0   = clock - r.start;
        for (uint64_t i = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < count; i += uint64_t(gridDim.x) * blockDim.x)
        {
            const uint64_t k    = k0 + i;
            if (k + 1 >= r.fade)
                y[i]                = yn[i];
            else
            {
                const float w       = float(double(k + 1) / double(r.fade));
                const float o       = y[i];
                y[i]                = fmaf(w, yn[i] - o, o);
            }
        }
    }
}

}   /* namespace b200conv */

#endif /* B200CONV_BATCH_FADE_CUH_ */

/*
 * b200conv::ConvolverBatch -- C++ RAII view of the C ABI (include/b200conv.h) for callers that
 * drive many lsp::dspu::Convolver-style instances together: N x init(), then ONE process() per
 * audio block for all instances x partitions.  Header only.
 */
#ifndef B200CONV_CONVOLVER_BATCH_H_
#define B200CONV_CONVOLVER_BATCH_H_

#include <b200conv.h>
#include <stddef.h>

namespace b200conv
{
    class ConvolverBatch
    {
        private:
            b200conv_batch_t   *pBatch;

        public:
            explicit ConvolverBatch(size_t instances, int device = -1): pBatch(NULL)
            {
                b200conv_create(&pBatch, device, instances);
            }
            ConvolverBatch(const ConvolverBatch &) = delete;
            ConvolverBatch & operator = (const ConvolverBatch &) = delete;
            ~ConvolverBatch()                       { b200conv_free(pBatch); }

            bool valid() const                      { return pBatch != NULL; }
            const char *error() const               { return b200conv_last_error(); }
            b200conv_batch_t *handle()              { return pBatch; }

            /** Convolver::init for instance idx */
            bool init(size_t idx, const float *data, size_t count, size_t rank, float phase)
                { return b200conv_init(pBatch, idx, data, count, rank, phase) == B200CONV_OK; }

            /** Same for a partition-range shard of a long impulse response */
            bool init_range(size_t idx, const float *data, size_t count, size_t rank, float phase, size_t part_offset)
                { return b200conv_init_range(pBatch, idx, data, count, rank, phase, part_offset) == B200CONV_OK; }

            /** Convolver::destroy for instance idx */
            void destroy(size_t idx)                { b200conv_destroy(pBatch, idx); }

            /** New impulse responses for running instances idx[0 .. count), crossfaded over fade samples */
            bool set_irs(size_t count, const size_t *idx, const float * const *data, const size_t *counts, size_t fade)
                { return b200conv_set_irs(pBatch, count, idx, data, counts, fade) == B200CONV_OK; }

            /** Samples of instance idx's crossfade still to come (0: not fading) */
            size_t fade_remaining(size_t idx) const { return b200conv_fade_remaining(pBatch, idx); }

            /** N x Convolver::process with host buffers, synchronous */
            bool process(float * const *dst, const float * const *src, size_t count)
                { return b200conv_process(pBatch, dst, src, count) == B200CONV_OK; }

            /** Same with device buffers [instances][stride], asynchronous on stream */
            bool process_device(float *dst, const float *src, size_t stride, size_t count, void *stream = NULL)
                { return b200conv_process_device(pBatch, dst, src, stride, count, stream) == B200CONV_OK; }

            /** Same with separate row pitches for the two matrices */
            bool process_device(float *dst, size_t dst_stride, const float *src, size_t src_stride, size_t count, void *stream)
                { return b200conv_process_device2(pBatch, dst, dst_stride, src, src_stride, count, stream) == B200CONV_OK; }

            bool sync()                             { return b200conv_sync(pBatch) == B200CONV_OK; }
            size_t data_size(size_t idx) const      { return b200conv_data_size(pBatch, idx); }
            size_t rank(size_t idx) const           { return b200conv_rank(pBatch, idx); }
            size_t instances() const                { return b200conv_instances(pBatch); }
    };
}

#endif /* B200CONV_CONVOLVER_BATCH_H_ */

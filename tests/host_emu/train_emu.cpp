// train_emu.cpp -- TEST INFRASTRUCTURE: the model-training kernels of redux_b200/csrc/redux_train.cuh run on the CPU.
// Every CTA runs its phases (zero, count, flush) thread by thread, each phase for all threads before the next, as the
// kernel's barriers order them.  Built by tests/test_train_models_emu.py with g++; compared there against the oracle.
// Not part of the product.
#include "cuda_shim.h"

#include <vector>

thread_local EmuIdx threadIdx, blockIdx, blockDim, gridDim;

// the threads of a CTA run one after another, so an atomic add is a plain add
static inline uint32_t atomicAdd(uint32_t *p, uint32_t v)
{
    const uint32_t old = *p;
    *p = old + v;
    return old;
}

#include "../../redux_b200/csrc/redux_train.cuh"

using namespace rdx;

extern "C" {

// Sub-histograms per CTA the kernel uses for symbol_bits s (0: counts go straight to the output row).
uint32_t emu_train_copies(uint32_t s) { return train_copies(s); }

// What redux_train_models_device enqueues (train_enqueue in redux_capi.cu), with `chunk` symbol positions per CTA
// (0: the library's kTrainChunk).  table: n_models start rows of 2^s + 1 entries; sample_model: the row of each
// sample (already checked); out: n_samples rows.
void emu_train(uint32_t s, uint32_t f, uint32_t chunk, const uint32_t *table, uint32_t n_models,
               const uint32_t *sample_model, const uint8_t *in, const uint64_t *in_off, uint64_t n_samples,
               uint64_t max_sample_len, uint32_t *out)
{
    const uint32_t nsym = (1u << s) + 1, fmax = (uint32_t)(((uint64_t)1 << f) - 1);
    std::vector<uint2> sample(n_samples);
    uint32_t max_room = 0;
    for (uint64_t i = 0; i < n_samples; ++i) {
        const uint32_t m = sample_model[i];
        uint64_t total = 0;
        for (uint32_t b = 0; b < nsym; ++b) total += table[(uint64_t)m * nsym + b];
        sample[i] = make_uint2(m, fmax - (uint32_t)total);
        if (sample[i].y > max_room) max_room = sample[i].y;
    }
    (void)n_models;
    TrainJob j;
    j.in = in; j.in_off = in_off; j.table = table; j.sample = sample.data(); j.out = out; j.n_samples = n_samples;
    j.s = s; j.nsym = nsym;
    j.chunk = chunk ? chunk : kTrainChunk;
    const uint64_t want = max_sample_len * 8 / s;
    const uint64_t limit = want < max_room ? want : max_room;
    j.chunks = (uint32_t)((limit + j.chunk - 1) / j.chunk);
    if (j.chunks == 0) j.chunks = 1;
    j.n_ctas = limit ? n_samples * j.chunks : 0;
    j.copies = train_copies(s);

    // train_init_kernel
    for (uint64_t i = 0; i < n_samples; ++i)
        for (uint32_t b = 0; b < nsym; ++b) out[i * nsym + b] = table[(uint64_t)sample[i].x * nsym + b];
    // train_count_kernel
    std::vector<uint32_t> hist(((size_t)j.copies << s) + 1);
    for (uint64_t cta = 0; cta < j.n_ctas; ++cta) {
        TrainRange r;
        if (!train_range(j, cta, &r)) continue;
        for (uint32_t t = 0; t < kTrainThreads; ++t) train_zero(j, hist.data(), t);
        for (uint32_t t = 0; t < kTrainThreads; ++t) train_count(j, r, hist.data(), t);
        for (uint32_t t = 0; t < kTrainThreads; ++t) train_flush(j, r, hist.data(), t);
    }
}

}  // extern "C"

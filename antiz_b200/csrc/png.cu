// PNG chunk runs (ATZ_SCAN_PNG_IDAT, ATZ_SCAN_APNG_FDAT): which of a shard's K1 candidates start a zlib stream split over consecutive
// IDAT or APNG fdAT chunks, and the lengths of its pieces in those chunks (common.cuh split_run).  Two passes, like K1: one thread per
// candidate counts the chunks of its run (nearly every candidate is rejected after the bytes before it), then one thread per run
// writes the lengths at the offsets the host has placed them (an exclusive sum of the counts: the output does not depend on thread
// timing).  The de-chunk copy of the runs' data into one buffer per stream is gather_kernel (scan.cu) with one job per chunk; the
// inflate is K2.
#include "common.cuh"

namespace atz {

// counts[k] = chunks of the run that starts at cand[k], RUN_FDAT set for an fdAT run (0: none, IDAT_FAR: the host walks it); the
// file is addressable in [lo, lim); flags: the context's ATZ_SCAN_* set
__global__ void __launch_bounds__(256) split_count_kernel(const uint8_t *file, uint64_t n, uint64_t lo, uint64_t lim, uint32_t flags, const uint32_t *cand, uint32_t ncand,
                                                          uint32_t *counts) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < ncand) counts[k] = split_run(file, n, lo, lim, cand[k], flags, nullptr, 0);
}

// run i starts at cand[which[i]]; its (counts[which[i]] & ~RUN_FDAT) piece lengths go to lens[at[i] ..]
__global__ void __launch_bounds__(256) split_write_kernel(const uint8_t *file, uint64_t n, uint64_t lo, uint64_t lim, uint32_t flags, const uint32_t *cand, const uint32_t *counts,
                                                          const uint32_t *which, const uint64_t *at, uint32_t nruns, uint32_t *lens) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < nruns) split_run(file, n, lo, lim, cand[which[i]], flags, lens + at[i], counts[which[i]] & ~RUN_FDAT);
}

cudaError_t launch_split_count(const uint8_t *file, uint64_t n, uint64_t lo, uint64_t lim, uint32_t flags, const uint32_t *cand, uint32_t ncand, uint32_t *counts, cudaStream_t s) {
    if (ncand) split_count_kernel<<<(ncand + 255) / 256, 256, 0, s>>>(file, n, lo, lim, flags, cand, ncand, counts);
    return cudaGetLastError();
}
cudaError_t launch_split_write(const uint8_t *file, uint64_t n, uint64_t lo, uint64_t lim, uint32_t flags, const uint32_t *cand, const uint32_t *counts, const uint32_t *which,
                               const uint64_t *at, uint32_t nruns, uint32_t *lens, cudaStream_t s) {
    if (nruns) split_write_kernel<<<(nruns + 255) / 256, 256, 0, s>>>(file, n, lo, lim, flags, cand, counts, which, at, nruns, lens);
    return cudaGetLastError();
}

} // namespace atz

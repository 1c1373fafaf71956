// PNG IDAT runs (ATZ_SCAN_PNG_IDAT): which of a shard's K1 candidates start a zlib stream split over consecutive IDAT chunks, and the
// lengths of those chunks (common.cuh idat_run).  Two passes, like K1: one thread per candidate counts the chunks of its run (nearly
// every candidate is rejected after the 8 bytes before it), then one thread per run writes the lengths at the offsets the host has
// placed them (an exclusive sum of the counts: the output does not depend on thread timing).  The de-chunk copy of the runs' data into
// one buffer per stream is gather_kernel (scan.cu) with one job per chunk; the inflate is K2.
#include "common.cuh"

namespace atz {

// counts[k] = chunks of the run that starts at cand[k] (0: none, IDAT_FAR: the host walks it); the file is addressable in [lo, lim)
__global__ void __launch_bounds__(256) idat_count_kernel(const uint8_t *file, uint64_t n, uint64_t lo, uint64_t lim, const uint32_t *cand, uint32_t ncand, uint32_t *counts) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < ncand) counts[k] = idat_run(file, n, lo, lim, cand[k], nullptr, 0);
}

// run i starts at cand[which[i]]; its counts[which[i]] chunk lengths go to lens[at[i] ..]
__global__ void __launch_bounds__(256) idat_write_kernel(const uint8_t *file, uint64_t n, uint64_t lo, uint64_t lim, const uint32_t *cand, const uint32_t *counts,
                                                         const uint32_t *which, const uint64_t *at, uint32_t nruns, uint32_t *lens) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < nruns) idat_run(file, n, lo, lim, cand[which[i]], lens + at[i], counts[which[i]]);
}

cudaError_t launch_idat_count(const uint8_t *file, uint64_t n, uint64_t lo, uint64_t lim, const uint32_t *cand, uint32_t ncand, uint32_t *counts, cudaStream_t s) {
    if (ncand) idat_count_kernel<<<(ncand + 255) / 256, 256, 0, s>>>(file, n, lo, lim, cand, ncand, counts);
    return cudaGetLastError();
}
cudaError_t launch_idat_write(const uint8_t *file, uint64_t n, uint64_t lo, uint64_t lim, const uint32_t *cand, const uint32_t *counts, const uint32_t *which,
                              const uint64_t *at, uint32_t nruns, uint32_t *lens, cudaStream_t s) {
    if (nruns) idat_write_kernel<<<(nruns + 255) / 256, 256, 0, s>>>(file, n, lo, lim, cand, counts, which, at, nruns, lens);
    return cudaGetLastError();
}

} // namespace atz

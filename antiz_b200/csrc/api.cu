// antiz_b200 C ABI (include/antiz_b200.h): device context, memory, the scan fold, the trial-wave scheduler.
// Everything that computes on bytes runs in the kernels of scan.cu / inflate.cu / chains.cu / deflate.cu; the host
// code here only orders work and folds fixed-size result records the way the reference's loops would
// (ZBuffSearcher::operator() main.cpp:205-246, findDeflateParams_stream main.cpp:561-602, testDeflateParams 685-715).
#include "../../include/antiz_b200.h"
#include "common.cuh"
#include <algorithm>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <map>
#include <mutex>
#include <thread>
#include <string>
#include <vector>
#include <chrono>

namespace atz {
// kernels (other translation units)
struct ChainTask { const uint8_t *in; uint32_t n; uint32_t hbits; uint32_t *list; uint32_t *idx; uint16_t *lsth; uint32_t *tmp; uint16_t *tmph; uint32_t chunk0, nchunks; };
struct AdlerJob { const uint8_t *in; uint32_t n; uint32_t *out; };
struct RowTask { const uint8_t *in; uint32_t n; const uint32_t *list, *idx; const uint16_t *lsth; const uint8_t *tmap; uint32_t *rows; uint32_t rlen, budget, chunk0, level, pbegin, visited_only; };
struct CopyJob { const uint8_t *src; uint8_t *dst; uint64_t n; };
struct DiffJob { const uint8_t *out; const uint8_t *orig; uint32_t cprime, c; uint32_t *pos; uint8_t *val; uint32_t cap; uint32_t *count; };
cudaError_t launch_deflate_trials(const TrialDesc *, TrialResult *, uint32_t, uint32_t *, const TrialOpts &, uint32_t *, uint8_t *, uint64_t, int, bool, cudaStream_t);
cudaError_t launch_build_chains(const ChainTask *, uint32_t, uint32_t, uint32_t *, uint32_t *, bool, cudaStream_t);
uint32_t chain_chunk_size();
cudaError_t launch_adler(const AdlerJob *, uint32_t, cudaStream_t);
cudaError_t launch_build_rows(const RowTask *, uint32_t, uint32_t, uint32_t *, int, cudaStream_t);
struct ResTask { const uint4 *rows; uint2 *out; uint32_t rlen, nice, jfull, jgood, maxd, chunk0, filtered; };
cudaError_t launch_resolve_rows(const ResTask *, uint32_t, uint32_t, cudaStream_t);
cudaError_t launch_gather(const CopyJob *, uint32_t, cudaStream_t);
cudaError_t launch_diff(const DiffJob *, uint32_t, cudaStream_t);
uint32_t scan_tiles_for(uint64_t lo, uint64_t hi);
cudaError_t launch_scan_count(const uint8_t *, uint64_t, uint64_t, uint64_t, uint32_t, uint32_t *, uint16_t *, uint32_t *, cudaStream_t);
cudaError_t launch_scan_write(const uint8_t *, uint64_t, uint64_t, const uint16_t *, const uint32_t *, uint32_t *, uint8_t *, uint32_t, cudaStream_t);
cudaError_t launch_inflate(const uint8_t *, const InflateJob *, InflateResult *, InflateResult *, uint32_t, uint32_t *, uint8_t *, uint64_t, uint64_t, int, int, cudaStream_t);
cudaError_t launch_split_count(const uint8_t *, uint64_t, uint64_t, uint64_t, uint32_t, const uint32_t *, uint32_t, uint32_t *, cudaStream_t);
cudaError_t launch_split_write(const uint8_t *, uint64_t, uint64_t, uint64_t, uint32_t, const uint32_t *, const uint32_t *, const uint32_t *, const uint64_t *, uint32_t, uint32_t *, cudaStream_t);
} // namespace atz
using namespace atz;

namespace {

struct Buf {   // grow-only device buffer
    void *p = nullptr; size_t cap = 0;
    cudaError_t ensure(size_t n) {
        if (n <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = n + n / 8 + 4096;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) { e = cudaMalloc(&p, n); want = n; }
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <class T> T *as() { return (T *)p; }
};

struct StreamRec {
    atz_stream s;
    const uint8_t *d_plain = nullptr;   // plaintext on the device (16 B aligned, ATZ_PAD slack); nullptr: another shard owns the stream
    const uint8_t *d_tmap = nullptr;    // token map of the original stream (common.cuh TM_*)
    const uint8_t *d_comp = nullptr;    // the stream's compressed bytes on the device (file image or the staging area of a sharded scan)
    uint32_t owner = 0;                 // shard that searches this stream (atz_host_partition)
    uint32_t adler = 0;
    std::vector<uint64_t> diff_off; std::vector<uint8_t> diff_val;
    std::vector<uint32_t> pieces;       // ATZ_SCAN_PNG_IDAT / ATZ_SCAN_APNG_FDAT: the piece lengths of a split stream (empty: an ordinary stream)
    uint32_t frame = 0;                 // bytes between two of its pieces: 12 (IDAT) or 16 (fdAT)
    uint64_t parent = 0; uint32_t depth = 0;   // a nested stream (ATZ_F_NESTED_DEPTH): atz_nested.parent and .depth; s.offset is relative to the parent's plaintext
    uint64_t span() const { return s.streamLength + (pieces.empty() ? 0 : (uint64_t)frame * (pieces.size() - 1)); }   // bytes from s.offset to the stream's end in the file
};

struct Params { uint8_t c, w, m, s = 0; };   // level, windowBits, memLevel, strategy (0 = Z_DEFAULT_STRATEGY: all the reference ever uses)

// One candidate the accept logic (scan_fold) can act on, as a shard exports it (atz_probe_export): the candidate inflated with its
// input cut at the end of its chunk (p_*) and, where that consumed the whole chunk, over the following chunks (c_*; c_status -1: none).
struct ProbeX {
    uint64_t off, avail, p_in, p_out, p_cap, c_in, c_out, c_cap;
    int32_t p_status, c_status; uint32_t p_adler, c_adler, local, type;
};
// A split stream (ATZ_SCAN_PNG_IDAT, ATZ_SCAN_APNG_FDAT) as a shard found it: the header offset, C and U of the de-chunked stream, its
// adler32 and header type, its piece lengths (the run's piece lengths up to the one that holds the stream's last byte, that one cut at
// C) and the framing bytes between two pieces (12: IDAT chunks, 16: fdAT chunks)
struct SplitX {
    uint64_t off, c, u; uint32_t adler, type; std::vector<uint32_t> pieces; uint32_t frame;
    uint64_t span() const { return c + (uint64_t)frame * (pieces.size() - 1); }
};
struct SplitDev { const uint8_t *comp, *plain, *tmap; };   // where the probing shard keeps a split stream's bytes
// State of a (possibly sharded) scan between atz_scan_shard and atz_scan_finish
struct ScanState {
    bool probed = false, resident = false; uint64_t S = 0, SLOT = 0, QS = 0; uint32_t shard = 0, nshards = 1;
    std::vector<uint32_t> cand; std::vector<uint8_t> ctype; std::vector<InflateJob> jobs; std::vector<InflateResult> res, cres;
    std::vector<const uint8_t *> big_plain, big_tmap;
    std::vector<std::vector<ProbeX>> px; std::vector<uint8_t> have;
    std::vector<std::vector<SplitX>> split; std::vector<SplitDev> split_dev;   // split streams of every shard; device bytes of this shard's
};

// coarse host-side stopwatch buckets (ATZ_DEBUG_HOST=1 prints them at the end of a search): per context, written by lane 0's thread only
struct HostDbg { bool lanes = false; std::chrono::steady_clock::time_point t0, t; double ms[8] = {0, 0, 0, 0, 0, 0, 0, 0}; double gpu = 0; };

inline uint64_t align_up(uint64_t v, uint64_t a) { return (v + a - 1) / a * a; }

// A search runs on up to ATZ_LANES lanes: one host thread + CUDA stream each, with its own scratch, arenas and counters, over a
// disjoint set of streams.  Every phase of a lane is bounded by that lane's longest stream (one warp per stream / per trial), so
// the tail of one lane's trial launch is filled by another lane's bucket sorts and row builds (DESIGN.md section 5a).
#define ATZ_LANES 4
struct TrialSlot {   // what one launch of the trial kernel needs: a stream, events around the launch, descriptors, results, per-warp scratch
    cudaStream_t stream = nullptr; cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    Buf descs, tres, symbuf, insmap, queue;
};
struct Lane {
    int id = 0; HostDbg *dbg = nullptr; cudaStream_t stream = nullptr; cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    Buf chains, recs, rtasks, restasks, tab, tasks, tmp_out, tmp_pos, tmp_val, tmp_cnt, djobs, queue;
    TrialSlot ts[2];   // [0] on the lane's stream; [1] on the side stream: the full-length reruns of a wave's prefix survivors, in the background (search_lane)
    Buf side_rtasks, side_restasks, side_queue, side_res;   // what a background launch needs of its own (kernel arguments, its resolved tables)
    atz_stats st{}; size_t budget = 0;
    std::vector<Buf *> bufs() { return {&chains, &recs, &rtasks, &restasks, &tab, &tasks, &tmp_out, &tmp_pos, &tmp_val, &tmp_cnt, &djobs, &queue,
                                        &ts[0].descs, &ts[0].tres, &ts[0].symbuf, &ts[0].insmap, &ts[0].queue, &ts[1].descs, &ts[1].tres, &ts[1].symbuf, &ts[1].insmap, &ts[1].queue, &side_rtasks, &side_restasks, &side_queue, &side_res}; }
};

} // namespace

struct atz_ctx {
    int device = 0; int nlanes_last = 1; cudaStream_t stream = nullptr; cudaEvent_t ev0 = nullptr, ev1 = nullptr, tev0 = nullptr, tev1 = nullptr;
    int sms = 148; size_t budget = 0;
    std::string err;
    int state = 0;   // 0 nothing, 1 loaded, 2 scanned, 3 searched
    uint32_t scan_flags = 0; bool scan_flags_fixed = false;   // ATZ_SCAN_*: the header set of the scan (atz_ctx_set_scan_flags, fixed by the first load)
    HostDbg dbg;
    // input: the file image.  d_file is the device address of file offset 0; bytes [r0, r1) are mapped there (everything after atz_load /
    // atz_load_device; after atz_attach only what this shard's scan and its owned streams need, uploaded from h_file on demand)
    Buf file; const uint8_t *d_file = nullptr; uint64_t n = 0;
    const uint8_t *h_file = nullptr; uint64_t r0 = 0, r1 = 0; Buf comp_extra;
    // scan
    Buf tile_counts, scan_masks, cand, ctype, jobs, jres, jres2, queue, total, idat_counts, idat_runs, idat_lens;
    ScanState sc;
    // streams
    std::vector<StreamRec> streams; Buf plain, plain2; std::vector<void *> plain_extra;   // stage-1 slots, stage-2 regions, retry rounds
    // nested streams of the last search (ATZ_F_NESTED_DEPTH), level by level; their plaintext and token maps live in nest_extra, the
    // scan buffer of a level and the probe slots in nest_scan / nest_slots (never ctx->plain: parents may live in its stage-1 slots)
    std::vector<StreamRec> nested; std::vector<void *> nest_extra; Buf nest_scan, nest_slots;
    // search
    Lane lane[ATZ_LANES];   // lane 0 runs on `stream` (the single-stream operators use it); 1.. have streams of lower priority
    Buf gather, cjobs;
    std::mutex err_mu;
    void set_err(const char *m) { std::lock_guard<std::mutex> g(err_mu); err = m; }
    // single-stream operators
    Buf op_in, op_orig, op_out, op_misc;
    atz_stats st{};
};

namespace {

#define CK(call)                                                                                         \
    do {                                                                                                 \
        cudaError_t e_ = (call);                                                                         \
        if (e_ != cudaSuccess) {                                                                         \
            char b_[512]; snprintf(b_, sizeof b_, "%s:%d %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); \
            ctx->set_err(b_); return e_ == cudaErrorMemoryAllocation ? ATZ_E_NOMEM : ATZ_E_CUDA;        \
        }                                                                                                \
    } while (0)

struct Phase {   // CUDA-event timing of a phase on the context stream / on a lane's stream
    cudaStream_t s; cudaEvent_t e0, e1; double *acc; int lane = -1; const char *what = ""; std::chrono::steady_clock::time_point h0; const HostDbg *dbg = nullptr;
    Phase(atz_ctx *c, double *a) : s(c->stream), e0(c->ev0), e1(c->ev1), acc(a) { cudaEventRecord(e0, s); }
    Phase(Lane &l, double *a, const char *w = "") : s(l.stream), e0(l.ev0), e1(l.ev1), acc(a), lane(l.id), what(w), dbg(l.dbg) { h0 = std::chrono::steady_clock::now(); cudaEventRecord(e0, s); }
    double stop() {
        cudaEventRecord(e1, s); cudaEventSynchronize(e1);
        float ms = 0; cudaEventElapsedTime(&ms, e0, e1); if (acc) *acc += ms; acc = nullptr;
        if (lane >= 0 && dbg && dbg->lanes) {   // host-clock timeline of the lanes' launches (ATZ_DEBUG_LANES=1)
            auto h1 = std::chrono::steady_clock::now();
            fprintf(stderr, "[lane %d] %-7s host %.2f .. %.2f ms  (gpu %.2f ms)\n", lane, what, std::chrono::duration<double, std::milli>(h0 - dbg->t0).count(),
                    std::chrono::duration<double, std::milli>(h1 - dbg->t0).count(), ms);
        }
        return ms;
    }
    ~Phase() { if (acc) stop(); }
};

int trial_slots(atz_ctx *ctx) { return ctx->sms * 24; }   // 3 CTAs x 8 warps per SM (80-register build); sparse launches use 2 x 8 at ~116 registers

// windowBits of a header type: the header's own for 0..23 (the reference's), 9 for CINFO 0 and 1 (ATZ_SCAN_SMALL_WINDOWS: zlib turns
// windowBits 8 into 9, and a CINFO 0 header is written over a window-9 stream)
inline int type_window(int offsetType) { return offsetType >= 24 ? 9 : 10 + offsetType / 4; }
#define ATZ_NTYPES 32
#define ATZ_NESTED_MAX 8   // deepest ATZ_F_NESTED_DEPTH

// ---- candidate order of the reference (main.cpp:487-602, 732-756) ----
void push_range(std::vector<Params> &v, int cmin, int cmax, int wmin, int wmax, int mmin, int mmax) {
    for (int w = wmax; w >= wmin; w--) for (int m = mmax; m >= mmin; m--) for (int c = cmax; c >= cmin; c--) v.push_back({(uint8_t)c, (uint8_t)w, (uint8_t)m});
}
void class_sequence(int offsetType, std::vector<Params> &v) {
    int w = type_window(offsetType);
    switch (offsetType % 4) {
    case 0: v.push_back({0, (uint8_t)w, 8}); v.push_back({1, (uint8_t)w, 8}); v.push_back({1, (uint8_t)w, 9});
            push_range(v, 1, 1, w, w, 1, 7); push_range(v, 2, 9, w, w, 1, 9); break;
    case 1: push_range(v, 2, 5, w, w, 8, 8); push_range(v, 2, 5, w, w, 1, 7); push_range(v, 2, 5, w, w, 9, 9);
            push_range(v, 1, 1, w, w, 1, 9); push_range(v, 6, 9, w, w, 1, 9); break;
    case 2: v.push_back({6, (uint8_t)w, 8}); v.push_back({6, (uint8_t)w, 9});
            push_range(v, 6, 6, w, w, 1, 7); push_range(v, 1, 5, w, w, 1, 9); push_range(v, 7, 9, w, w, 1, 9); break;
    default: push_range(v, 7, 9, w, w, 8, 8); push_range(v, 7, 9, w, w, 1, 7); push_range(v, 7, 9, w, w, 9, 9);
             push_range(v, 1, 6, w, w, 1, 9); break;
    }
}
// (window 9, types 24..31: the whole grid 15..10, window 9 is not in it)
void brute_sequence(int offsetType, std::vector<Params> &v) {
    int w = type_window(offsetType);
    if (w == 10) push_range(v, 1, 9, 11, 15, 1, 9);
    else if (w == 15) push_range(v, 1, 9, 10, 14, 1, 9);
    else { push_range(v, 1, 9, 10, w - 1, 1, 9); push_range(v, 1, 9, w + 1, 15, 1, 9); }
}


// ATZ_F_STRATEGIES (extension): the other zlib strategies at the header's window, memLevel 9..1, levels high to low -
// Z_FILTERED (1) only where it differs from the default (deflate_slow levels), Z_FIXED (4) everywhere, Z_RLE (3) and
// Z_HUFFMAN_ONLY (2) once per memLevel (their output does not depend on the level)
void strategy_sequence(int offsetType, std::vector<Params> &v) {
    const int w = type_window(offsetType);
    for (int m = 9; m >= 1; m--) for (int c = 9; c >= 4; c--) v.push_back({(uint8_t)c, (uint8_t)w, (uint8_t)m, 1});
    for (int m = 9; m >= 1; m--) for (int c = 9; c >= 1; c--) v.push_back({(uint8_t)c, (uint8_t)w, (uint8_t)m, 4});
    for (int m = 9; m >= 1; m--) v.push_back({1, (uint8_t)w, (uint8_t)m, 3});
    for (int m = 9; m >= 1; m--) v.push_back({1, (uint8_t)w, (uint8_t)m, 2});
}

// ---- host-side scan logic (pure functions; also exported for CPU tests as atz_host_*) ----
struct ProbeRec { int32_t status; uint64_t total_in, total_out, in_at_outcap; };
struct Acc { uint64_t off, tin, tout; uint32_t cand; bool via_cont; };

// chunk list of searchInfile (main.cpp:405-415): first read S bytes, then S-1 new bytes behind the kept last byte;
// the loop runs until a read comes up short, so a file of exactly S + k(S-1) bytes gets a trailing 1-byte chunk.
// The byte the reference keeps for the overlap is `rBuffer[f.gcount() - 1]` (main.cpp:408, 413): the last byte of chunk 0, but -
// since later chunks are read into rBuffer + 1 - the SECOND TO LAST byte of every other chunk.  So chunk k >= 2 does not start with
// file[start_k] but with file[start_k - 1]; positions keep their nominal offsets.  What follows from that is reproduced: a header is
// looked for in (file[start_k - 1], file[start_k + 1]) at offset start_k, a candidate there inflates those bytes, and a continuation
// entering chunk k >= 2 sees that byte repeated (atz_scan_shard, InflateJob::flags).
void chunk_list(uint64_t N, uint64_t S, std::vector<uint64_t> &cstart, std::vector<uint64_t> &clen) {
    cstart.clear(); clen.clear();
    uint64_t pos = std::min(S, N); bool eof = N < S;
    cstart.push_back(0); clen.push_back(pos);
    while (!eof) { uint64_t got = std::min(S - 1, N - pos); cstart.push_back(pos - 1); clen.push_back(got + 1); pos += got; eof = got < S - 1; }
}

// ZBuffSearcher::operator() replayed over per-candidate result records (main.cpp:205-246, SURVEY.md A.1).
//   probe[k]   : candidate k inflated with its input cut at the end of its chunk (avail[k] bytes)
//   cont_of[k] : index into cont[] of the run over "rest of chunk, then the following chunks each starting with the
//                duplicated overlap byte" (only for candidates that consumed their whole chunk), or -1
void scan_fold(const std::vector<uint64_t> &cstart, const std::vector<uint64_t> &clen, const uint32_t *cand, uint32_t ncand, const ProbeRec *probe,
               const uint64_t *avail, const int32_t *cont_of, const ProbeRec *cont, std::vector<Acc> &acc) {
    const size_t nch = cstart.size();
    bool need_more = false, carried_finished = false; uint32_t carried = 0; uint64_t carried_consumed = 0, last_chunk_offset = 0;
    size_t ci = 0;   // next candidate index
    for (size_t c = 0; c < nch; c++) {
        const uint64_t start = cstart[c], len = clen[c];
        uint64_t i = 0;
        if (need_more) {   // refillInput with the new chunk (main.cpp:207-217)
            const ProbeRec *vr = cont_of[carried] >= 0 ? &cont[cont_of[carried]] : nullptr;
            // a decoder left in BAD state (error exactly at the end of its chunk) has no continuation run: it consumes nothing
            int vstatus = vr ? vr->status : INF_DATA_ERROR; uint64_t vin = vr ? vr->total_in : carried_consumed, vout = vr ? vr->total_out : 0;
            if (carried_finished) {   // DONE / BAD: inflate() returns at once, avail_in stays len
                if (vstatus == INF_END) { acc.push_back({last_chunk_offset, vin, vout, carried, true}); i = 0; }
                need_more = (len == 0);
            } else {
                bool event = (vstatus == INF_END || vstatus == INF_DATA_ERROR || vstatus == INF_NEED_DICT);
                uint64_t e = vin - carried_consumed;
                if (event && vin >= carried_consumed && e <= len) {
                    if (vstatus == INF_END) { acc.push_back({last_chunk_offset, vin, vout, carried, true}); i = e; }
                    need_more = (e == len); carried_finished = true;
                } else { need_more = true; carried_consumed += len; }
            }
        }
        if (!need_more && len >= 2) {
            const uint64_t redlen = len - 1;
            while (ci < ncand && cand[ci] < start + i) ci++;
            while (i < redlen && ci < ncand && cand[ci] < start + redlen) {
                const uint32_t k = (uint32_t)ci; const uint64_t f = cand[k]; i = f - start;
                const ProbeRec &r = probe[k];
                if (r.in_at_outcap <= 16) { i++; ci++; continue; }               // main.cpp:229
                if (r.status == INF_END) {                                       // main.cpp:234-237
                    acc.push_back({f, r.total_in, r.total_out, k, false});
                    i += r.total_in;
                    while (ci < ncand && cand[ci] < start + i) ci++;
                    continue;
                }
                if (r.total_in == avail[k]) {                                    // avail_in == 0, main.cpp:238-239
                    need_more = true; last_chunk_offset = f; carried = k; carried_consumed = avail[k];
                    carried_finished = (r.status != INF_NEED_INPUT);
                    ci++;
                    break;
                }
                i++; ci++;
            }
        }
        // the skip position is per chunk (main.cpp:206): the next chunk starts at its own i = 0
        if (c + 1 < nch) { while (ci > 0 && cand[ci - 1] >= cstart[c + 1]) ci--; }
    }
}

// Lanes of a search (atz_search_shard): streams sorted by plaintext length; lane 0 (highest stream priority) takes the longest
// ones - its launches are the critical path, a warp per stream - and each following lane a larger share of shorter streams,
// whose sorts and row builds fill the tails of the lanes ahead.  The per-stream results do not depend on the partition.
// Measured: lanes pay where the host's share of a step is large - many small streams: +36 % on configs[3]; on long streams the
// latency-bound trial warps of one lane are slowed by the row builds of another by as much as the overlap gains, or more - so
// the default is 1 lane unless the mean stream is under 32 KB.  forced > 0 overrides the count (test hook ATZ_LANES).
// part[l] = indices into ulen[], ascending; returns the number of lanes.
int lane_partition(const uint64_t *ulen, uint32_t n, int forced, std::vector<std::vector<uint32_t>> &part) {
    uint64_t tot = 0; for (uint32_t k = 0; k < n; k++) tot += ulen[k];
    const bool lanes_pay = n && tot / n < 32768;
    int nl = lanes_pay ? (int)std::min<size_t>(ATZ_LANES, std::max<size_t>(1, n / 16)) : 1;
    if (forced > 0) nl = std::min(ATZ_LANES, forced);
    part.assign(nl, std::vector<uint32_t>());
    if (nl == 1) { part[0].resize(n); for (uint32_t k = 0; k < n; k++) part[0][k] = k; return nl; }
    std::vector<uint32_t> ord(n); for (uint32_t k = 0; k < n; k++) ord[k] = k;
    std::stable_sort(ord.begin(), ord.end(), [&](uint32_t a, uint32_t b) { return ulen[a] > ulen[b]; });
    static const double kShare[ATZ_LANES][ATZ_LANES] = {{1, 1, 1, 1}, {0.35, 1, 1, 1}, {0.2, 0.55, 1, 1}, {0.15, 0.4, 0.7, 1}};   // cumulative share of the bytes
    uint64_t acc = 0; int l = 0;
    for (uint32_t k : ord) {
        while (l + 1 < nl && (double)acc >= kShare[nl - 1][l] * (double)tot) l++;
        part[l].push_back(k); acc += ulen[k];
    }
    for (auto &v : part) std::sort(v.begin(), v.end());
    return nl;
}

// Static partition of the accepted streams over the shards of a multi-GPU run (SURVEY.md 8e).  Trials per stream are not known
// before the search, so the load of a shard is its plaintext bytes (+ a per-stream constant: many tiny streams cost more than their
// bytes); the streams that turn out to need the whole --brute-window grid are spread like the others, in proportion to their length.
//   probed_by == nullptr: longest plaintext first, each to the least loaded shard (ties: the lowest shard);
//   probed_by[k] = shard whose chunk range stream k starts in (a sharded scan): the plaintext is already resident there, so a stream
//   stays where it was probed unless that shard holds more than 2 % above the mean; the excess moves to the least loaded shards,
//   streams of at most 64 KB first (what moves is inflated again by its new owner: a launch as long as its longest stream).
// Deterministic: every context computes the same owners from the same stream list.
void stream_partition(const uint64_t *ulen, const uint32_t *probed_by, uint32_t n, uint32_t nshards, uint32_t *owner) {
    if (nshards <= 1) { for (uint32_t k = 0; k < n; k++) owner[k] = 0; return; }
    auto cost = [&](uint32_t k) { return ulen[k] + 4096; };
    std::vector<uint32_t> ord(n); for (uint32_t k = 0; k < n; k++) ord[k] = k;
    std::stable_sort(ord.begin(), ord.end(), [&](uint32_t a, uint32_t b) { return ulen[a] > ulen[b]; });
    std::vector<uint64_t> load(nshards, 0);
    auto least = [&]() { uint32_t best = 0; for (uint32_t g = 1; g < nshards; g++) if (load[g] < load[best]) best = g; return best; };
    if (!probed_by) {
        for (uint32_t k : ord) { const uint32_t g = least(); owner[k] = g; load[g] += cost(k); }
        return;
    }
    uint64_t total = 0;
    for (uint32_t k = 0; k < n; k++) { owner[k] = probed_by[k] < nshards ? probed_by[k] : 0; load[owner[k]] += cost(k); total += cost(k); }
    const uint64_t mean = total / nshards, hi = mean + mean / 50;
    for (int pass = 0; pass < 2; pass++)
        for (uint32_t k : ord) {
            const uint32_t src = owner[k];
            if (load[src] <= hi) continue;
            if ((pass == 0) != (ulen[k] <= 65536)) continue;
            const uint32_t dst = least();
            if (dst == src || load[dst] + cost(k) > hi) continue;
            owner[k] = dst; load[src] -= cost(k); load[dst] += cost(k);
        }
}

struct ChainKey { uint32_t stream, hbits; };
inline bool needs_chain(const Params &p) { return p.c != 0 && p.s != 2 && p.s != 3; }     // level 0, deflate_huff and deflate_rle look at no hash chain

// Generic plaintext view used by the trial machinery (streams of a scan, or operator inputs)
struct PlainView { const uint8_t *d_in; uint32_t n; const uint8_t *d_orig; uint32_t c; uint32_t adler; const uint8_t *d_tmap = nullptr; };

struct TrialReq { uint32_t view; Params prm; uint8_t store; uint8_t *d_out; uint32_t out_cap; uint8_t want_rec = 0, want_res = 0, phase1 = 0, reserve_whole = 0, all_rows = 0; };   // all_rows: deflate_slow rows at every position, not only where the original's parse looked   // reserve_whole: size a new row table for the whole stream (it is likely to be extended)   // want_rec: 0 no rows, 1 first-block prefix, 2 whole stream; want_res: resolved table (levels 4-9)

struct RowRef { const uint4 *rows = nullptr; uint32_t rlen = 0, budget = 0, cap = 0; bool vis = false; };   // vis: rows only at the positions the original's parse visited   // cap: positions the allocation has room for
// chains and row tables of a batch of views, dense: [view][memLevel 1..9] and [view][memLevel][0 = deflate_slow, 1..3 = deflate_fast level]
struct ChainState {
    std::vector<ChainRef> chains; std::vector<RowRef> rows; uint64_t chain_used = 0, rec_used = 0;
    struct Want { uint32_t budget = 0, rlen = 0, reserve = 0; bool all = false; }; std::vector<Want> want; std::vector<uint32_t> touched;
    void init(size_t nviews) { if (chains.size() < nviews * 9) { chains.resize(nviews * 9, ChainRef{nullptr, nullptr, nullptr, nullptr, 0, 0}); rows.resize(nviews * 36); want.resize(nviews * 36); } }
    ChainRef &chain(uint32_t view, uint32_t m) { return chains[(size_t)view * 9 + (m - 1)]; }
    static uint32_t rkey(uint32_t view, uint32_t m, uint32_t level) { return (view * 9 + (m - 1)) * 4 + level; }
};
static const uint16_t kChainBudget[10] = {0, 4, 8, 32, 16, 32, 128, 256, 1024, 4096};
static const uint16_t kNice[10] = {0, 8, 16, 32, 16, 32, 128, 128, 258, 258};   // Z/deflate.c:131-143

static inline double gpu_ms_sum(const Lane &L) { return L.st.ms_chains + L.st.ms_rows + L.st.ms_trials + L.st.ms_diff; }
// host time (wall minus GPU-event time) since the previous mark goes to bucket k (lane 0 only: a debugging aid)
static inline void host_mark(const Lane &L, int k) {
    if (L.id != 0 || !L.dbg) return;
    HostDbg &D = *L.dbg;
    auto now = std::chrono::steady_clock::now(); double g = gpu_ms_sum(L);
    if (k >= 0) D.ms[k] += std::chrono::duration<double, std::milli>(now - D.t).count() - (g - D.gpu);
    D.t = now; D.gpu = g;
}

#define TR_PENDING (-1)   /* host side only: the result of a trial launched on the side stream, not collected yet */
struct Launched { TrialSlot *x = nullptr; std::vector<uint32_t> idx; std::vector<TrialDesc> descs; std::vector<TrialResult> tmp; bool dense = false, pending = false; };

// One launch of the trial kernel for the requests `sel` (indices into reqs) on slot X; chains, rows and resolved tables exist.
// Does not wait: collect_trials() does.  dense_mode: 1 = the 80-register build, 0 = the full-register build, -1 = by count.
int launch_trials(atz_ctx *ctx, Lane &L, TrialSlot &X, const std::vector<PlainView> &views, const std::vector<TrialReq> &reqs, const std::vector<uint32_t> &sel,
                  const std::vector<const uint2 *> &res_of, const TrialOpts &opts, ChainState &cs, int dense_mode, Launched &ln) {
    ln.x = &X; ln.pending = false; ln.idx.clear();
    if (sel.empty()) return ATZ_OK;
    // most expensive first (queue order).  expected cost: bytes the trial will parse (a phase-1 trial stops after its first block of
    // lit_bufsize symbols, ~3.5 B each) x cycles per byte of the path it will take (stored / row-driven / bucket walks)
    std::vector<float> cost(sel.size());
    for (size_t i = 0; i < sel.size(); i++) {
        const TrialReq &r = reqs[sel[i]]; const PlainView &v = views[r.view];
        float bytes = (float)v.n;
        if (r.phase1) bytes = std::min(bytes, 3.5f * (float)(64u << r.prm.m));
        const bool rows = r.want_rec != 0 && (r.prm.c >= 4 || v.d_tmap != nullptr);
        const float per = r.prm.c == 0 ? 0.05f : r.prm.c <= 3 ? (rows ? 1.5f : 4.f) : (r.want_res ? 1.f : rows ? 2.5f : 2.5f + 0.5f * (r.prm.c - 4));
        cost[i] = bytes * per;
    }
    // Queue order: by expected cost, most expensive first (the length of a launch is at least that of its longest trial).
    std::vector<uint32_t> order(sel.size());
    for (uint32_t i = 0; i < order.size(); i++) order[i] = i;
    std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return cost[a] > cost[b]; });
    ln.idx.resize(sel.size()); ln.descs.resize(sel.size());
    uint32_t max_fast_n = 0;
    for (size_t k = 0; k < order.size(); k++) {
        const uint32_t ri = sel[order[k]]; ln.idx[k] = ri;
        const TrialReq &r = reqs[ri]; const PlainView &v = views[r.view];
        TrialDesc d{}; d.in = v.d_in; d.orig = v.d_orig; d.out = r.d_out; d.n = v.n; d.c = v.c; d.out_cap = r.out_cap; d.adler = v.adler;
        d.level = r.prm.c; d.wbits = r.prm.w; d.memlevel = r.prm.m; d.store = r.store; d.phase1 = r.phase1; d.strategy = r.prm.s;
        if (needs_chain(r.prm)) {
            d.ch = cs.chain(r.view, r.prm.m);
            const RowRef *it = &cs.rows[ChainState::rkey(r.view, r.prm.m, r.prm.c >= 4 ? 0u : (uint32_t)r.prm.c)];
            if (it->rows && it->budget >= kChainBudget[r.prm.c]) {
                d.ch.rec = it->rows; d.ch.rlen = it->rlen; d.ch.rbudget = it->budget;
                if (r.prm.c <= 3) d.tmap = v.d_tmap; else { d.res = res_of[ri]; if (d.res) d.tmap = v.d_tmap; }
            }
        }
        if (r.prm.c >= 1 && r.prm.c <= 3 && needs_chain(r.prm)) max_fast_n = std::max(max_fast_n, v.n);
        ln.descs[k] = d;
    }
    const uint32_t nt = (uint32_t)ln.descs.size();
    uint64_t stride = align_up((uint64_t)max_fast_n / 8 + 64, 256);     // inserted map: one bit per plaintext position
    const bool dense = dense_mode >= 0 ? dense_mode != 0 : (int)nt > ctx->sms * 16;
    int slots = dense ? ctx->sms * 24 : ctx->sms * 16;     // (64 registers / 32 warps per SM was measured: 763 vs 665 ms per step on the 128 MB mixed corpus)
    if (max_fast_n) {   // bound the inserted-map scratch
        uint64_t lim = std::max<uint64_t>((uint64_t)8 << 30, L.budget / 8);
        while (slots > 64 && (uint64_t)slots * stride > lim) slots /= 2;
    }
    const int ctas = (int)std::min<uint32_t>((uint32_t)slots, nt);     // one warp per CTA (launch_deflate_trials)
    CK(X.queue.ensure(64));
    CK(X.symbuf.ensure((size_t)ctas * 32768 * 4));
    if (max_fast_n) CK(X.insmap.ensure((size_t)ctas * stride));
    CK(X.descs.ensure(nt * sizeof(TrialDesc)));
    CK(X.tres.ensure(nt * sizeof(TrialResult)));
    CK(cudaMemcpyAsync(X.descs.p, ln.descs.data(), nt * sizeof(TrialDesc), cudaMemcpyHostToDevice, X.stream));
    CK(cudaMemsetAsync(X.queue.p, 0, 4, X.stream));
    CK(cudaEventRecord(X.ev0, X.stream));
    CK(launch_deflate_trials(X.descs.as<TrialDesc>(), X.tres.as<TrialResult>(), nt, X.queue.as<uint32_t>(), opts, X.symbuf.as<uint32_t>(),
                             X.insmap.as<uint8_t>(), stride, ctas, dense, X.stream));
    CK(cudaEventRecord(X.ev1, X.stream));
    ln.tmp.resize(nt);     // (copied back by collect_trials: a device-to-pageable copy queued here would block the host until the kernel is done)
    ln.dense = dense; ln.pending = true;
    return ATZ_OK;
}
// Wait for a launch and hand its results out by request index.
int collect_trials(atz_ctx *ctx, Lane &L, Launched &ln, std::vector<TrialResult> &out) {
    if (!ln.pending) return ATZ_OK;
    ln.pending = false;
    TrialSlot &X = *ln.x;
    CK(cudaStreamSynchronize(X.stream));
    CK(cudaGetLastError());
    CK(cudaMemcpy(ln.tmp.data(), X.tres.p, ln.tmp.size() * sizeof(TrialResult), cudaMemcpyDeviceToHost));
    float ms = 0; CK(cudaEventElapsedTime(&ms, X.ev0, X.ev1));
    L.st.ms_trials += ms; L.st.kernel_launches++; L.st.n_trial_kernels++;
    if (ms > L.st.ms_trials_max_kernel) L.st.ms_trials_max_kernel = ms;
    const uint32_t nt = (uint32_t)ln.tmp.size();
    for (uint32_t k = 0; k < nt; k++) out[ln.idx[k]] = ln.tmp[k];
    if (L.dbg && L.dbg->lanes) fprintf(stderr, "[lane %d] trials%s %u collected at host %.2f ms (gpu %.2f ms)\n", L.id, &X == &L.ts[1] ? " (side)" : "", nt,
                               std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - L.dbg->t0).count(), ms);
    if (getenv("ATZ_DEBUG_TRIALS")) {   // which trials a launch waits for: kilocycles by (level, status), and the slowest few
        const std::vector<TrialDesc> &descs = ln.descs; const std::vector<TrialResult> &tmp = ln.tmp;
        struct Agg { uint64_t n = 0, kc = 0, kf = 0, mx = 0; }; std::map<std::pair<int, int>, Agg> agg;
        std::vector<uint32_t> o(nt); for (uint32_t i = 0; i < nt; i++) o[i] = i;
        for (uint32_t i = 0; i < nt; i++) { Agg &a = agg[{descs[i].level, tmp[i].status}]; a.n++; a.kc += tmp[i].kcycles; a.kf += tmp[i].kcycles_flush; a.mx = std::max<uint64_t>(a.mx, tmp[i].kcycles); }
        std::sort(o.begin(), o.end(), [&](uint32_t a, uint32_t b) { return tmp[a].kcycles > tmp[b].kcycles; });
        fprintf(stderr, "[trials] launch of %u (%s%s)\n", nt, ln.dense ? "dense" : "sparse", &X == &L.ts[1] ? ", side stream" : "");
        for (auto &kv : agg) fprintf(stderr, "   level %d status %d: n %llu sum %llu kcyc (flush %llu) max %llu\n", kv.first.first, kv.first.second, (unsigned long long)kv.second.n,
                                     (unsigned long long)kv.second.kc, (unsigned long long)kv.second.kf, (unsigned long long)kv.second.mx);
        for (uint32_t q = 0; q < std::min<uint32_t>(6, nt); q++) { const TrialDesc &d = descs[o[q]]; const TrialResult &r = tmp[o[q]];
            fprintf(stderr, "   slow: l%d w%d m%d n %u c %u phase1 %u rows %d res %d tmap %d -> status %d consumed %u kcyc %u (flush %u)\n", d.level, d.wbits, d.memlevel, d.n, d.c, d.phase1,
                    d.ch.rec ? (int)d.ch.rlen : 0, d.res != nullptr, d.tmap != nullptr, r.status, r.in_consumed, r.kcycles, r.kcycles_flush); }
    }
    L.st.gpu_trials += nt;
    return ATZ_OK;
}

// Build missing chains, row and resolved tables, run one kernel launch of trials, bring the results back.
// `bg`: where given, nothing is waited for: tables and trials are queued on the lane's side stream (with kernel-argument buffers and a
// resolved-table arena of their own) and the launch is left pending in *bg until the caller collects it (collect_trials).  Every
// request's bucket lists must exist already (its candidate has been through a foreground launch).
int run_trials(atz_ctx *ctx, Lane &L, const std::vector<PlainView> &views, const std::vector<TrialReq> &reqs, const TrialOpts &opts,
               ChainState &cs, std::vector<TrialResult> &out, bool allow_dense = true, Launched *bg = nullptr) {
    uint64_t &chain_used = cs.chain_used;
    cs.init(views.size());
    out.assign(reqs.size(), TrialResult{});
    if (reqs.empty()) return ATZ_OK;
    host_mark(L, 0);   // caller: building requests, folding results
    const cudaStream_t S = bg ? L.ts[1].stream : L.stream;
    Buf &B_rtasks = bg ? L.side_rtasks : L.rtasks, &B_restasks = bg ? L.side_restasks : L.restasks, &B_queue = bg ? L.side_queue : L.queue;
    if (bg) for (auto &r : reqs) if (needs_chain(r.prm) && !cs.chain(r.view, r.prm.m).list) { ctx->set_err("background launch without bucket lists"); return ATZ_E_STATE; }
    // ---- chains ----
    std::vector<ChainTask> tasks;
    for (auto &r : reqs) {
        if (!needs_chain(r.prm)) continue;
        ChainKey k{r.view, (uint32_t)r.prm.m + 7};
        if (cs.chain(r.view, r.prm.m).list) continue;
        const PlainView &v = views[r.view];
        uint64_t np = v.n >= 3 ? v.n - 2 : 0;
        uint64_t o_list = align_up(chain_used, 256), o_idx = align_up(o_list + 4 * (np + 32), 256), o_cnt = align_up(o_idx + 4 * (np + 32), 256);
        uint64_t end = align_up(o_cnt + 2 * (np + 32), 256);
        // a stream whose bucket lists do not fit the arena (hundreds of MB of plaintext against the default budget): its candidates of this
        // hash size are not run and count as "no match" - the stream stays un-recompressed instead of failing the whole file
        if (end > L.chains.cap) { ctx->set_err("chain arena exhausted for one stream: left un-recompressed (raise atz_ctx_set_budget)"); continue; }
        chain_used = end;
        uint8_t *b = L.chains.as<uint8_t>();
        ChainRef cr{(const uint32_t *)(b + o_list), (const uint32_t *)(b + o_idx), (const uint16_t *)(b + o_cnt), nullptr, 0, 0};
        cs.chain(r.view, r.prm.m) = cr;
        tasks.push_back(ChainTask{v.d_in, v.n, k.hbits, (uint32_t *)cr.list, (uint32_t *)cr.idx, (uint16_t *)cr.lsth, nullptr, nullptr, 0, 0});
    }
    CK(L.queue.ensure(64));
    if (!tasks.empty()) {
        // scratch: pass-1 output (u32 position + u16 hash per entry) of the two-pass tasks, chunk histograms, per-task digit bases
        const uint32_t CH = chain_chunk_size();
        uint64_t scratch = 0; uint32_t chunks = 0; bool any_two = false;
        for (auto &t : tasks) {
            uint64_t np = t.n >= 3 ? t.n - 2 : 0;
            t.chunk0 = chunks; t.nchunks = (uint32_t)((np + CH - 1) / CH); chunks += t.nchunks;
            if (t.hbits > 8) { any_two = true; scratch = align_up(scratch, 256) + 4 * (np + 64); scratch = align_up(scratch, 256) + 2 * (np + 64); }
        }
        const uint64_t o_hist = align_up(scratch, 256), o_dbase = o_hist + (uint64_t)chunks * 1024;
        CK(L.tab.ensure(o_dbase + tasks.size() * 1024 + 256));
        { uint64_t o = 0; uint8_t *tb = L.tab.as<uint8_t>();
          for (auto &t : tasks) if (t.hbits > 8) {
              uint64_t np = t.n >= 3 ? t.n - 2 : 0;
              o = align_up(o, 256); t.tmp = (uint32_t *)(tb + o); o += 4 * (np + 64);
              o = align_up(o, 256); t.tmph = (uint16_t *)(tb + o); o += 2 * (np + 64);
          } }
        if (chunks) {
        CK(L.tasks.ensure(tasks.size() * sizeof(ChainTask)));
        CK(cudaMemcpyAsync(L.tasks.p, tasks.data(), tasks.size() * sizeof(ChainTask), cudaMemcpyHostToDevice, L.stream));
        Phase ph(L, &L.st.ms_chains, "chains");
        CK(launch_build_chains(L.tasks.as<ChainTask>(), (uint32_t)tasks.size(), chunks, (uint32_t *)(L.tab.as<uint8_t>() + o_hist), (uint32_t *)(L.tab.as<uint8_t>() + o_dbase), any_two, L.stream));
        ph.stop(); L.st.kernel_launches += any_two ? 6 : 3;
        }
        CK(cudaGetLastError());
    }
    host_mark(L, 1);
    // ---- row tables (deflate.cu build_rows_kernel): level 0 = deflate_slow rows of one hash size, 1..3 = deflate_fast rows
    // under the original stream's token map ----
    {
        typedef ChainState::Want Want;
        cs.touched.clear();
        const int force = getenv("ATZ_FORCE_REC") ? atoi(getenv("ATZ_FORCE_REC")) : -1;   // test hook: 0 = never, 2 = always whole-stream tables
        for (auto &r : reqs) {
            int wr = force >= 0 ? force : r.want_rec;
            if (!needs_chain(r.prm) || !wr || !cs.chain(r.view, r.prm.m).list) continue;
            const PlainView &v = views[r.view]; uint32_t np = v.n >= 3 ? v.n - 2 : 0;
            uint32_t rlen;
            if (r.prm.c >= 4) {
                uint32_t pre = (uint32_t)std::min<uint64_t>(np, (uint64_t)4 * (64u << r.prm.m) + 2048);   // ~ the first block (lit_bufsize symbols)
                rlen = wr >= 2 ? np : pre;
            } else {
                if (!v.d_tmap || v.n <= 2048) continue;
                rlen = v.n - 1024;     // the token map's insert classes are exact only clear of the end of the stream (deflate.cu run_fast)
            }
            const uint32_t key = ChainState::rkey(r.view, r.prm.m, r.prm.c >= 4 ? 0u : (uint32_t)r.prm.c);
            Want &w = cs.want[key];
            if (w.budget == 0) cs.touched.push_back(key);
            w.budget = std::max<uint32_t>(w.budget, kChainBudget[r.prm.c]); w.rlen = std::max(w.rlen, rlen);
            if (r.reserve_whole && r.prm.c >= 4) w.reserve = np;
            if (r.all_rows) w.all = true;
        }
        std::vector<RowTask> rt; uint32_t chunks = 0;
        for (uint32_t key : cs.touched) {
            const Want w = cs.want[key]; cs.want[key] = Want{};
            const uint32_t kview = key / 36, km = (key / 4) % 9 + 1, klevel = key % 4;
            const PlainView &v = views[kview];
            RowRef &rr = cs.rows[key];
            const bool all_env = getenv("ATZ_ALL_ROWS") != nullptr;
            const bool want_vis = klevel == 0 && v.d_tmap != nullptr && !w.all && !all_env;
            if (w.rlen == 0 || (rr.rows && rr.rlen >= w.rlen && rr.budget >= w.budget && (want_vis || !rr.vis))) continue;
            const ChainRef &cr = cs.chain(kview, km);
            // a longer table for the same key: the rows that exist are kept (they looked at least as far down the chains) and only
            // the rest is built - for deflate_slow restricted to the positions the original parse visited, when its token map is known
            uint32_t pbegin = 0, vis = 0, cap = rr.cap; uint32_t *rp = (uint32_t *)rr.rows;
            const bool keep = rr.rows && rr.budget >= w.budget && klevel == 0 && (want_vis || !rr.vis);   // (a table of visited positions only is not extended into a full one: rebuilt)
            if (klevel == 0) vis = want_vis;
            if (keep) pbegin = rr.rlen & ~31u;
            if (!(keep && rr.cap >= w.rlen)) {     // no room to extend in place: a new allocation (and the kept rows copied over)
                cap = std::max(w.rlen, w.reserve);
                uint64_t o = align_up(cs.rec_used, 256), end = o + 32ull * cap;
                if (end > L.recs.cap) { cap = w.rlen; end = o + 32ull * cap; }
                if (end > L.recs.cap) continue;                                            // arena full: those trials walk their chains
                cs.rec_used = end;
                rp = (uint32_t *)(L.recs.as<uint8_t>() + o);
                if (pbegin) CK(cudaMemcpyAsync(rp, rr.rows, 32ull * pbegin, cudaMemcpyDeviceToDevice, S));
            }
            rt.push_back(RowTask{v.d_in, v.n, cr.list, cr.idx, cr.lsth, v.d_tmap, rp, w.rlen, w.budget, chunks, klevel, pbegin, vis});
            chunks += (w.rlen - pbegin + 31) / 32;
            rr.rows = (const uint4 *)rp; rr.rlen = std::max(w.rlen, keep ? rr.rlen : 0u); rr.budget = w.budget; rr.cap = cap; rr.vis = vis != 0;
        }
        if (!rt.empty()) {
            CK(B_rtasks.ensure(rt.size() * sizeof(RowTask))); CK(B_queue.ensure(64));
            CK(cudaMemcpyAsync(B_rtasks.p, rt.data(), rt.size() * sizeof(RowTask), cudaMemcpyHostToDevice, S));      // (pageable source: staged by the runtime before the call returns)
            CK(cudaMemsetAsync(B_queue.p, 0, 4, S));
            int ctas = (int)std::min<uint32_t>((uint32_t)ctx->sms * 8, (chunks + 7) / 8);
            if (bg) { CK(launch_build_rows(B_rtasks.as<RowTask>(), (uint32_t)rt.size(), chunks, B_queue.as<uint32_t>(), ctas, S)); }
            else {
                Phase ph(L, &L.st.ms_rows, "rows");
                CK(launch_build_rows(B_rtasks.as<RowTask>(), (uint32_t)rt.size(), chunks, B_queue.as<uint32_t>(), ctas, S));
                ph.stop();
            }
            L.st.kernel_launches++;
            CK(cudaGetLastError());
        }
    }
    host_mark(L, 2);
    // ---- resolved tables for full-length level 4-9 trials (deflate.cu resolve_rows_kernel) ----
    std::vector<const uint2 *> res_of(reqs.size(), nullptr);
    const uint64_t res_mark = cs.rec_used;   // resolved tables live for this launch only (a background launch has an arena of its own for them)
    {
        std::vector<ResTask> rt; uint32_t chunks = 0;
        const int force = getenv("ATZ_FORCE_RES") ? atoi(getenv("ATZ_FORCE_RES")) : -1;   // test hook: 0 = never, 1 = whenever rows exist
        uint64_t bg_used = 0;
        if (bg) {
            uint64_t need = 0;
            for (size_t i = 0; i < reqs.size(); i++) {
                const TrialReq &r = reqs[i];
                if (r.prm.c < 4 || !needs_chain(r.prm) || !(force >= 0 ? force : r.want_res)) continue;
                const RowRef *it = &cs.rows[ChainState::rkey(r.view, r.prm.m, 0u)];
                if (it->rows && it->budget >= kChainBudget[r.prm.c]) need = align_up(need, 256) + 8ull * it->rlen;
            }
            if (need && need <= L.budget / 4) { if (L.side_res.ensure(need + 256) != cudaSuccess) { cudaGetLastError(); L.side_res.cap = 0; L.side_res.p = nullptr; } }
        }
        for (size_t i = 0; i < reqs.size(); i++) {
            const TrialReq &r = reqs[i];
            if (r.prm.c < 4 || !needs_chain(r.prm) || !(force >= 0 ? force : r.want_res)) continue;
            const RowRef *it = &cs.rows[ChainState::rkey(r.view, r.prm.m, 0u)];
            if (!it->rows || it->budget < kChainBudget[r.prm.c]) continue;
            uint2 *out;
            if (bg) {
                uint64_t o = align_up(bg_used, 256), end = o + 8ull * it->rlen;
                if (end > L.side_res.cap) continue;
                bg_used = end; out = (uint2 *)(L.side_res.as<uint8_t>() + o);
            } else {
                uint64_t o = align_up(cs.rec_used, 256), end = o + 8ull * it->rlen;
                if (end > L.recs.cap) continue;
                cs.rec_used = end; out = (uint2 *)(L.recs.as<uint8_t>() + o);
            }
            uint32_t jfull = 0; while ((1u << (jfull + 1)) <= kChainBudget[r.prm.c]) jfull++;
            rt.push_back(ResTask{it->rows, out, it->rlen, kNice[r.prm.c], jfull, jfull >= 2 ? jfull - 2 : 0, (1u << r.prm.w) - 262u, chunks, r.prm.s == 1 ? 1u : 0u});
            chunks += (it->rlen + 255) / 256;
            res_of[i] = out;
        }
        if (!rt.empty()) {
            CK(B_restasks.ensure(rt.size() * sizeof(ResTask)));
            CK(cudaMemcpyAsync(B_restasks.p, rt.data(), rt.size() * sizeof(ResTask), cudaMemcpyHostToDevice, S));
            if (bg) { CK(launch_resolve_rows(B_restasks.as<ResTask>(), (uint32_t)rt.size(), chunks, S)); }
            else {
                Phase ph(L, &L.st.ms_rows, "rows");
                CK(launch_resolve_rows(B_restasks.as<ResTask>(), (uint32_t)rt.size(), chunks, S));
                ph.stop();
            }
            L.st.kernel_launches++;
            CK(cudaGetLastError());
        }
    }
    host_mark(L, 3);
    // ---- trials (a request whose bucket lists could not be allocated is answered "size gate failed": the fold ignores it) ----
    std::vector<uint32_t> all; all.reserve(reqs.size());
    for (uint32_t i = 0; i < reqs.size(); i++) {
        if (needs_chain(reqs[i].prm) && !cs.chain(reqs[i].view, reqs[i].prm.m).list) { out[i].status = TR_SIZE; continue; }
        all.push_back(i);
    }
    if (bg) {
        int rc = launch_trials(ctx, L, L.ts[1], views, reqs, all, res_of, opts, cs, allow_dense ? -1 : 0, *bg); if (rc) return rc;
        for (uint32_t i : all) out[i].status = TR_PENDING;
        host_mark(L, 4);
        return ATZ_OK;
    }
    Launched main;
    { int rc = launch_trials(ctx, L, L.ts[0], views, reqs, all, res_of, opts, cs, allow_dense ? -1 : 0, main); if (rc) return rc; }
    host_mark(L, 4);
    { int rc = collect_trials(ctx, L, main, out); if (rc) return rc; }
    cs.rec_used = res_mark;
    host_mark(L, 5);
    return ATZ_OK;
}

TrialOpts make_opts(const atz_options *o, bool compare) {
    TrialOpts t{};
    t.compare = compare ? 1 : 0;
    const int burst_env = getenv("ATZ_BURST") ? atoi(getenv("ATZ_BURST")) : 1;   // test hook: 0 = serial parse loops only
    t.burst = burst_env ? 1 : 0;
    if (!o) { t.shortcut = 0xffffffffu; t.bail_below = 0; t.sizediff = 0xffffffffu; t.cut_mismatch = 0xffffffffu; return t; }
    t.shortcut = (uint32_t)std::min<uint64_t>(o->shortcutLength, 0xfffffff0u);
    uint64_t thr = o->shortcutLength - o->recompTresh;   // unsigned wrap on purpose (main.cpp:649)
    t.bail_below = (uint32_t)std::min<uint64_t>(thr, 0xffffffffu);
    t.sizediff = (uint32_t)std::min<uint64_t>(o->sizediffTresh, 0xfffffff0u);
    t.cut_mismatch = (o->flags & ATZ_F_EXACT_RECORDS) ? 0xffffffffu : (uint32_t)std::min<uint64_t>(std::max(o->recompTresh, o->mismatchTol), 0xfffffff0u);
    return t;
}

int rec_arena_for(atz_ctx *ctx, Lane &L, uint64_t worst_bytes) {
    uint64_t want = std::min<uint64_t>(worst_bytes, L.budget / 2);
    want = std::max<uint64_t>(want, 1 << 20);
    if (L.recs.cap >= want) return ATZ_OK;
    L.recs.release();
    cudaError_t e = cudaMalloc(&L.recs.p, want);
    while (e != cudaSuccess && want > (64u << 20)) { cudaGetLastError(); want /= 2; e = cudaMalloc(&L.recs.p, want); }
    if (e != cudaSuccess) { cudaGetLastError(); L.recs.p = nullptr; L.recs.cap = 0; return ATZ_OK; }   // optional accelerator
    L.recs.cap = want;
    return ATZ_OK;
}
int chain_arena_for(atz_ctx *ctx, Lane &L, uint64_t worst_bytes) {
    uint64_t want = std::min<uint64_t>(worst_bytes, L.budget / 2);
    want = std::max<uint64_t>(want, 1 << 20);
    if (L.chains.cap >= want) return ATZ_OK;
    L.chains.release();
    cudaError_t e = cudaMalloc(&L.chains.p, want);
    while (e != cudaSuccess && want > (64u << 20)) { cudaGetLastError(); want /= 2; e = cudaMalloc(&L.chains.p, want); }
    if (e != cudaSuccess) { ctx->set_err("cannot allocate chain arena"); return ATZ_E_NOMEM; }
    L.chains.cap = want;
    return ATZ_OK;
}
inline uint64_t chain_bytes(uint64_t n) { uint64_t np = n + 32; return 3 * 256 + 10 * np + 768; }

} // namespace

// =================================================================================================
extern "C" {

const char *atz_version(void) { return "antiz_b200 0.1 (sm_100a; AntiZ 0.1.6-git semantics, zlib 1.2.8 bit-exact)"; }
const char *atz_last_error(atz_ctx *ctx) { return ctx ? ctx->err.c_str() : "no context"; }

int atz_ctx_create(int device, atz_ctx **out) {
    if (!out) return ATZ_E_ARG;
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0 || device < 0 || device >= ndev) { cudaGetLastError(); return ATZ_E_NO_DEVICE; }
    if (cudaSetDevice(device) != cudaSuccess) return ATZ_E_NO_DEVICE;
    atz_ctx *ctx = new atz_ctx();
    ctx->device = device;
    cudaDeviceProp pr;
    if (cudaGetDeviceProperties(&pr, device) != cudaSuccess) { delete ctx; return ATZ_E_NO_DEVICE; }
    if (pr.major < 10) { delete ctx; return ATZ_E_NO_DEVICE; }   // kernels are built for sm_100a only
    ctx->sms = pr.multiProcessorCount;
    int prio_least = 0, prio_greatest = 0; cudaDeviceGetStreamPriorityRange(&prio_least, &prio_greatest);
    if (cudaStreamCreateWithPriority(&ctx->stream, cudaStreamNonBlocking, prio_greatest) != cudaSuccess) { delete ctx; return ATZ_E_CUDA; }
    cudaEventCreate(&ctx->ev0); cudaEventCreate(&ctx->ev1); cudaEventCreate(&ctx->tev0); cudaEventCreate(&ctx->tev1);
    for (int l = 0; l < ATZ_LANES; l++) {   // lane 0 gets the longest streams and the highest priority (atz_search_shard)
        Lane &L = ctx->lane[l]; L.id = l;
        const int prio = std::min(prio_least, prio_greatest + l);
        if (l == 0) { L.stream = ctx->stream; L.ev0 = ctx->ev0; L.ev1 = ctx->ev1; }
        else {
            if (cudaStreamCreateWithPriority(&L.stream, cudaStreamNonBlocking, prio) != cudaSuccess) { cudaGetLastError(); atz_ctx_destroy(ctx); return ATZ_E_CUDA; }
            cudaEventCreate(&L.ev0); cudaEventCreate(&L.ev1);
        }
        L.ts[0].stream = L.stream;
        if (cudaStreamCreateWithPriority(&L.ts[1].stream, cudaStreamNonBlocking, prio) != cudaSuccess) { cudaGetLastError(); atz_ctx_destroy(ctx); return ATZ_E_CUDA; }
        for (int k = 0; k < 2; k++) { cudaEventCreate(&L.ts[k].ev0); cudaEventCreate(&L.ts[k].ev1); }
    }
    size_t fr = 0, tot = 0; cudaMemGetInfo(&fr, &tot);
    ctx->budget = (size_t)(fr * 0.6);
    *out = ctx;
    return ATZ_OK;
}
void atz_ctx_destroy(atz_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    Buf *all[] = {&ctx->file, &ctx->tile_counts, &ctx->scan_masks, &ctx->cand, &ctx->ctype, &ctx->jobs, &ctx->jres, &ctx->queue, &ctx->jres2, &ctx->total, &ctx->idat_counts, &ctx->idat_runs, &ctx->idat_lens, &ctx->plain, &ctx->plain2,
                  &ctx->gather, &ctx->cjobs, &ctx->comp_extra, &ctx->op_in, &ctx->op_orig, &ctx->op_out, &ctx->op_misc, &ctx->nest_scan, &ctx->nest_slots};
    for (Buf *b : all) b->release();
    for (void *q : ctx->plain_extra) cudaFree(q);
    for (void *q : ctx->nest_extra) cudaFree(q);
    for (int l = 0; l < ATZ_LANES; l++) {
        Lane &L = ctx->lane[l];
        if (L.ts[1].stream) { cudaStreamSynchronize(L.ts[1].stream); cudaStreamDestroy(L.ts[1].stream); }
        for (int k = 0; k < 2; k++) { if (L.ts[k].ev0) cudaEventDestroy(L.ts[k].ev0); if (L.ts[k].ev1) cudaEventDestroy(L.ts[k].ev1); }
        for (Buf *b : L.bufs()) b->release();
        if (l && L.stream) { cudaStreamSynchronize(L.stream); cudaStreamDestroy(L.stream); if (L.ev0) cudaEventDestroy(L.ev0); if (L.ev1) cudaEventDestroy(L.ev1); }
    }
    cudaEventDestroy(ctx->ev0); cudaEventDestroy(ctx->ev1); cudaEventDestroy(ctx->tev0); cudaEventDestroy(ctx->tev1); cudaStreamDestroy(ctx->stream);
    delete ctx;
}
int atz_ctx_set_budget(atz_ctx *ctx, uint64_t bytes) { if (!ctx || bytes < (1u << 20)) return ATZ_E_ARG; ctx->budget = bytes; return ATZ_OK; }
int atz_ctx_set_scan_flags(atz_ctx *ctx, uint32_t flags) {
    if (!ctx || (flags & ~(uint32_t)(ATZ_SCAN_SMALL_WINDOWS | ATZ_SCAN_PNG_IDAT | ATZ_SCAN_APNG_FDAT))) return ATZ_E_ARG;
    if (ctx->scan_flags_fixed) { ctx->set_err("atz_ctx_set_scan_flags: the context has already loaded a file"); return ATZ_E_STATE; }
    ctx->scan_flags = flags;
    return ATZ_OK;
}

static void drop_nested(atz_ctx *ctx) {
    ctx->nested.clear();
    for (void *q : ctx->nest_extra) cudaFree(q);
    ctx->nest_extra.clear();
}
static void reset_scan(atz_ctx *ctx) {
    drop_nested(ctx);
    ctx->st = atz_stats{}; ctx->streams.clear(); ctx->state = 0; ctx->sc = ScanState{}; ctx->scan_flags_fixed = true;
}
static int load_common(atz_ctx *ctx, const void *src, uint64_t n, cudaMemcpyKind kind) {
    if (!ctx || !src || n == 0) return ATZ_E_ARG;
    if (n >= 0xffffff00ull) return ATZ_E_TOO_LARGE;
    cudaSetDevice(ctx->device);
    reset_scan(ctx);
    CK(ctx->file.ensure(n + ATZ_PAD));
    Phase ph(ctx, &ctx->st.ms_h2d);
    CK(cudaMemcpyAsync(ctx->file.p, src, n, kind, ctx->stream));
    CK(cudaMemsetAsync(ctx->file.as<uint8_t>() + n, 0, ATZ_PAD, ctx->stream));
    ph.stop();
    ctx->d_file = ctx->file.as<uint8_t>(); ctx->n = n; ctx->h_file = nullptr; ctx->r0 = 0; ctx->r1 = n; ctx->state = 1;
    return ATZ_OK;
}
int atz_load(atz_ctx *ctx, const uint8_t *file, uint64_t n) { return load_common(ctx, file, n, cudaMemcpyHostToDevice); }
int atz_load_device(atz_ctx *ctx, const void *dev_file, uint64_t n) { return load_common(ctx, dev_file, n, cudaMemcpyDeviceToDevice); }
int atz_attach(atz_ctx *ctx, const uint8_t *file, uint64_t n) {
    if (!ctx || !file || n == 0) return ATZ_E_ARG;
    if (n >= 0xffffff00ull) return ATZ_E_TOO_LARGE;
    reset_scan(ctx);
    ctx->h_file = file; ctx->n = n; ctx->d_file = nullptr; ctx->r0 = ctx->r1 = 0; ctx->state = 1;
    return ATZ_OK;
}
// Make file bytes [a, b) addressable as ctx->d_file + offset.  After atz_attach this uploads the range (start rounded down to 256 so
// that the 16-byte loads of the scan kernel stay aligned) and replaces whatever range was mapped before.
static int ensure_range(atz_ctx *ctx, uint64_t a, uint64_t b) {
    b = std::min(b, ctx->n);
    if (a >= ctx->r0 && b <= ctx->r1 && ctx->d_file) return ATZ_OK;
    if (!ctx->h_file) { ctx->set_err("file range not resident"); return ATZ_E_STATE; }
    const uint64_t a0 = a & ~255ull, len = b > a0 ? b - a0 : 0;
    CK(ctx->file.ensure(len + ATZ_PAD));
    Phase ph(ctx, &ctx->st.ms_h2d);
    if (len) CK(cudaMemcpyAsync(ctx->file.p, ctx->h_file + a0, len, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemsetAsync(ctx->file.as<uint8_t>() + len, 0, ATZ_PAD, ctx->stream));
    ph.stop();
    ctx->d_file = (const uint8_t *)((uintptr_t)ctx->file.p - (uintptr_t)a0); ctx->r0 = a0; ctx->r1 = a0 + len;
    return ATZ_OK;
}

// ---------------------------------------------------------------------------------------------
// Phase 1.  The file is cut into the reference's chunks (chunk_list); shard g of G probes the candidates that start in its
// contiguous range of chunks (K1 + K2), exports one fixed-size record per candidate the accept logic can act on, and after the
// records of all shards have been put together (atz_probe_import; nothing to do for G = 1) every context replays the sequential
// accept logic over them (scan_fold: cheap, deterministic, replicated), partitions the accepted streams (atz_host_partition) and
// makes sure the plaintext of the streams it owns is resident.  SURVEY.md 8(e); main.cpp:392-420, 205-246.
static int run_inflate(atz_ctx *ctx, const uint8_t *base, std::vector<InflateJob> &jv, std::vector<InflateResult> &rv, std::vector<InflateResult> &cv, uint8_t *arena,
                       uint64_t S, double *acc) {
    if (jv.empty()) return ATZ_OK;
    const int iwpc = 4; const int islots = ctx->sms * 16;
    uint32_t nj = (uint32_t)jv.size();
    int wpc = iwpc, ctas;
    if ((int)nj <= ctx->sms * 4) { wpc = 1; ctas = (int)nj; } else ctas = (int)std::min<uint32_t>((uint32_t)(islots / wpc), (nj + wpc - 1) / wpc);
    CK(ctx->jobs.ensure(nj * sizeof(InflateJob))); CK(ctx->jres.ensure(nj * sizeof(InflateResult))); CK(ctx->jres2.ensure(nj * sizeof(InflateResult)));
    CK(cudaMemcpyAsync(ctx->jobs.p, jv.data(), nj * sizeof(InflateJob), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemsetAsync(ctx->queue.p, 0, 4, ctx->stream));
    Phase ph(ctx, acc);
    CK(launch_inflate(base, ctx->jobs.as<InflateJob>(), ctx->jres.as<InflateResult>(), ctx->jres2.as<InflateResult>(), nj, ctx->queue.as<uint32_t>(), arena,
                      S, S, ctas, wpc, ctx->stream));
    ph.stop(); ctx->st.kernel_launches++;
    CK(cudaGetLastError());
    rv.resize(nj); cv.resize(nj);
    CK(cudaMemcpyAsync(rv.data(), ctx->jres.p, nj * sizeof(InflateResult), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(cv.data(), ctx->jres2.p, nj * sizeof(InflateResult), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return ATZ_OK;
}

// ---- ATZ_SCAN_PNG_IDAT, ATZ_SCAN_APNG_FDAT ----
#define SPLIT_FLAGS (ATZ_SCAN_PNG_IDAT | ATZ_SCAN_APNG_FDAT)
struct RunBytes { uint64_t off; const uint32_t *len; size_t npieces; uint64_t total; uint32_t frame; };   // a run's pieces in the file: piece k+1 starts frame bytes after piece k
// The pieces of every run put together in one new device buffer (freed with plain_extra at the next scan), each run at at[i] with ATZ_PAD
// zeroed bytes behind it: one gather launch over the file image for the runs inside the mapped range, host copies from the attached file
// for the others.
static int dechunk(atz_ctx *ctx, const std::vector<RunBytes> &runs, uint8_t *&base, std::vector<uint64_t> &at) {
    at.resize(runs.size()); uint64_t tot = 0;
    for (size_t i = 0; i < runs.size(); i++) { at[i] = tot; tot = align_up(tot + runs[i].total + ATZ_PAD, 256); }
    void *q = nullptr; CK(cudaMalloc(&q, tot + ATZ_PAD)); ctx->plain_extra.push_back(q); base = (uint8_t *)q;
    CK(cudaMemsetAsync(q, 0, tot + ATZ_PAD, ctx->stream));
    std::vector<CopyJob> cj; std::vector<uint8_t> stage;
    for (size_t i = 0; i < runs.size(); i++) {
        const RunBytes &r = runs[i];
        const bool mapped = ctx->d_file && r.off >= ctx->r0 && r.off + r.total + (uint64_t)r.frame * (r.npieces - 1) <= ctx->r1;
        if (!mapped && !ctx->h_file) { ctx->set_err("chunk run outside the resident file range"); return ATZ_E_STATE; }
        if (!mapped) stage.resize(r.total);
        uint64_t src = r.off, dst = 0;
        for (size_t k = 0; k < r.npieces; k++) {
            if (mapped) cj.push_back(CopyJob{ctx->d_file + src, base + at[i] + dst, r.len[k]});
            else memcpy(stage.data() + dst, ctx->h_file + src, r.len[k]);
            dst += r.len[k]; src += r.len[k] + r.frame;
        }
        if (!mapped && r.total) { CK(cudaMemcpyAsync(base + at[i], stage.data(), r.total, cudaMemcpyHostToDevice, ctx->stream)); CK(cudaStreamSynchronize(ctx->stream)); }
    }
    if (!cj.empty()) {
        CK(ctx->cjobs.ensure(cj.size() * sizeof(CopyJob)));
        CK(cudaMemcpyAsync(ctx->cjobs.p, cj.data(), cj.size() * sizeof(CopyJob), cudaMemcpyHostToDevice, ctx->stream));
        CK(launch_gather(ctx->cjobs.as<CopyJob>(), (uint32_t)cj.size(), ctx->stream)); ctx->st.kernel_launches++;
        CK(cudaStreamSynchronize(ctx->stream));
    }
    return ATZ_OK;
}

// The split streams of this shard: the K1 candidates (cand, type: K1's own list) that start an IDAT or fdAT run (png.cu; the kinds the
// scan flags enable), each inflated by K2 over its run's pieces put together; a stream that ends there beyond its first piece and is
// longer than 16 bytes is recorded (SplitX) with its plaintext and token map left resident, like a probed ordinary stream's.
static int probe_split_runs(atz_ctx *ctx, const std::vector<uint32_t> &cand, const std::vector<uint8_t> &type) {
    ScanState &sc = ctx->sc; const uint64_t N = ctx->n; const uint32_t flags = ctx->scan_flags;
    const uint32_t nc = (uint32_t)cand.size();
    std::vector<uint32_t> which, cnt, frame; std::vector<uint64_t> at; std::vector<uint32_t> lens;   // run i: candidate which[i], cnt[i] lengths at lens[at[i]]
    if (nc) {
        std::vector<uint32_t> counts(nc);
        Phase ph(ctx, &ctx->st.ms_scan);
        CK(ctx->idat_counts.ensure((size_t)nc * 4));
        CK(launch_split_count(ctx->d_file, N, ctx->r0, ctx->r1, flags, ctx->cand.as<uint32_t>(), nc, ctx->idat_counts.as<uint32_t>(), ctx->stream)); ctx->st.kernel_launches++;
        CK(cudaMemcpyAsync(counts.data(), ctx->idat_counts.p, (size_t)nc * 4, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        std::vector<uint32_t> dw; std::vector<uint64_t> dat; uint64_t tot = 0;
        for (uint32_t k = 0; k < nc; k++) if (counts[k] && counts[k] != IDAT_FAR) { dw.push_back(k); dat.push_back(tot); tot += counts[k] & ~RUN_FDAT; }
        lens.resize(tot);
        if (!dw.empty()) {
            CK(ctx->idat_runs.ensure(dw.size() * 12)); CK(ctx->idat_lens.ensure(tot * 4));
            uint64_t *d_at = ctx->idat_runs.as<uint64_t>(); uint32_t *d_which = (uint32_t *)(d_at + dw.size());   // (the 8-byte offsets first: aligned)
            CK(cudaMemcpyAsync(d_at, dat.data(), dw.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
            CK(cudaMemcpyAsync(d_which, dw.data(), dw.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
            CK(launch_split_write(ctx->d_file, N, ctx->r0, ctx->r1, flags, ctx->cand.as<uint32_t>(), ctx->idat_counts.as<uint32_t>(), d_which, d_at, (uint32_t)dw.size(),
                                  ctx->idat_lens.as<uint32_t>(), ctx->stream));
            ctx->st.kernel_launches++;
            CK(cudaMemcpyAsync(lens.data(), ctx->idat_lens.p, tot * 4, cudaMemcpyDeviceToHost, ctx->stream));
        }
        ph.stop();
        // runs that leave the resident range (atz_attach): walked again over the whole attached file
        size_t j = 0;
        for (uint32_t k = 0; k < nc; k++) {
            uint32_t m = counts[k];
            if (m == IDAT_FAR) {
                if (!ctx->h_file) { ctx->set_err("chunk run outside the resident file range"); return ATZ_E_STATE; }
                m = split_run(ctx->h_file, N, 0, N, cand[k], flags, nullptr, 0);
                if (!m) continue;
                at.push_back(lens.size()); lens.resize(lens.size() + (m & ~RUN_FDAT));
                split_run(ctx->h_file, N, 0, N, cand[k], flags, lens.data() + at.back(), m & ~RUN_FDAT);
            } else if (j < dw.size() && dw[j] == k) at.push_back(dat[j++]);
            else continue;
            which.push_back(k); cnt.push_back(m & ~RUN_FDAT); frame.push_back(m & RUN_FDAT ? 16 : 12);
        }
    }
    const size_t nr = which.size();
    std::vector<RunBytes> runs(nr);
    for (size_t i = 0; i < nr; i++) {
        RunBytes r{cand[which[i]], lens.data() + at[i], cnt[i], 0, frame[i]};
        for (size_t k = 0; k < cnt[i]; k++) r.total += r.len[k];
        runs[i] = r;
    }
    sc.split[sc.shard].clear(); sc.split_dev.clear();
    if (!nr) return ATZ_OK;
    uint8_t *comp = nullptr; std::vector<uint64_t> cat;
    { int rc = dechunk(ctx, runs, comp, cat); if (rc) return rc; }
    // K2 over the de-chunked runs: the plaintext length is not known, so a region that turns out too small is enlarged and the job rerun
    std::vector<size_t> todo(nr); std::vector<uint64_t> cap(nr);
    for (size_t i = 0; i < nr; i++) { todo[i] = i; cap[i] = align_up(std::max<uint64_t>(4 * 8192, 5 * runs[i].total) + 16384, 256); }
    std::vector<InflateResult> fin(nr); std::vector<const uint8_t *> plain(nr), tmap(nr);
    while (!todo.empty()) {
        uint64_t arena = 0; std::vector<InflateJob> bj(todo.size()); std::vector<InflateResult> br, bc;
        for (size_t t = 0; t < todo.size(); t++) {
            const size_t i = todo[t];
            bj[t] = InflateJob{cat[i], runs[i].total, runs[i].total, arena, cap[i], 0, 0};
            arena = align_up(arena + cap[i] + ATZ_PAD, 256); bj[t].tmap_off = arena; arena = align_up(arena + cap[i] + 64, 256);
        }
        void *q = nullptr; CK(cudaMalloc(&q, arena + ATZ_PAD)); ctx->plain_extra.push_back(q);
        CK(cudaMemsetAsync(q, 0, arena + ATZ_PAD, ctx->stream));
        { int rc = run_inflate(ctx, comp, bj, br, bc, (uint8_t *)q, sc.S, &ctx->st.ms_inflate_probe); if (rc) return rc; }
        std::vector<size_t> again;
        for (size_t t = 0; t < todo.size(); t++) {
            const size_t i = todo[t];
            if (br[t].status == INF_OUT_FULL) {
                const uint64_t lim = 1032 * runs[i].total + 65536;
                if (cap[i] >= lim) { ctx->set_err("inflate output exceeds the deflate expansion bound"); return ATZ_E_CUDA; }
                cap[i] = std::min<uint64_t>(align_up(cap[i] * 6, 256), align_up(lim, 256)); again.push_back(i);
            } else { fin[i] = br[t]; plain[i] = (uint8_t *)q + bj[t].out_off; tmap[i] = (uint8_t *)q + bj[t].tmap_off; }
        }
        todo.swap(again);
    }
    for (size_t i = 0; i < nr; i++) {
        const InflateResult &r = fin[i]; const uint64_t C = r.total_in;
        if (r.status != INF_END || C <= runs[i].len[0] || C <= 16) continue;
        SplitX x{runs[i].off, C, r.total_out, r.adler, type[which[i]], {}, runs[i].frame};
        for (uint64_t k = 0, got = 0; got < C; k++) { const uint64_t l = std::min<uint64_t>(runs[i].len[k], C - got); x.pieces.push_back((uint32_t)l); got += l; }
        sc.split[sc.shard].push_back(std::move(x)); sc.split_dev.push_back(SplitDev{comp + cat[i], plain[i], tmap[i]});
    }
    return ATZ_OK;
}

int atz_scan_shard(atz_ctx *ctx, uint64_t chunksize, uint32_t shard, uint32_t nshards) {
    if (!ctx || nshards == 0 || shard >= nshards) return ATZ_E_ARG;
    if (ctx->state < 1) return ATZ_E_STATE;
    if (chunksize < 2) return ATZ_E_ARG;
    cudaSetDevice(ctx->device);
    const uint64_t N = ctx->n, S = chunksize;
    drop_nested(ctx);     // (their bytes point into the plaintext freed below)
    ctx->streams.clear(); ctx->state = 1;
    ScanState &sc = ctx->sc; sc = ScanState{};
    sc.S = S; sc.shard = shard; sc.nshards = nshards; sc.px.assign(nshards, std::vector<ProbeX>()); sc.have.assign(nshards, 0);
    sc.split.assign(nshards, std::vector<SplitX>());
    std::vector<uint64_t> cstart, clen;
    chunk_list(N, S, cstart, clen);
    const size_t nch = cstart.size();
    std::vector<uint64_t> suffix(nch + 1, 0);
    for (size_t c = nch; c-- > 0;) suffix[c] = suffix[c + 1] + clen[c];
    // this shard's chunks [c0, c1) and the file positions [f0, f1) whose candidates it probes (chunk of f = f / (S-1): the
    // overlap byte of two chunks is a start position of the later one only, main.cpp:411-414 + redlen main.cpp:220)
    const size_t c0 = nch * shard / nshards, c1 = nch * (shard + 1) / nshards;
    const uint64_t f0 = c0 == 0 ? 0 : cstart[c0], f1 = c1 >= nch ? N : cstart[c1];
    CK(ctx->tile_counts.ensure((size_t)scan_tiles_for(f0, f1) * 4 + 64)); CK(ctx->total.ensure(64)); CK(ctx->queue.ensure(64));
    CK(ctx->scan_masks.ensure((size_t)scan_tiles_for(f0, f1) * 8192 + 64));
    for (void *q : ctx->plain_extra) cudaFree(q);
    ctx->plain_extra.clear();
    const uint64_t Q = 8192, QS = align_up(Q + ATZ_PAD, 256), QT = align_up(Q + 64, 256), SLOT = QS + QT;
    sc.QS = QS; sc.SLOT = SLOT;
    std::vector<uint32_t> &cand = sc.cand; std::vector<uint8_t> &ctype = sc.ctype;
    std::vector<InflateJob> &jobs = sc.jobs; std::vector<InflateResult> &res = sc.res, &cres = sc.cres;
    std::vector<uint32_t> k1cand; std::vector<uint8_t> k1type;    // SPLIT_FLAGS: K1's own candidates (the real file bytes, no chunk-start fix-up)
    // a continuation (a stream that runs over the end of its chunk) reads the following chunks: map `extra` of them behind the
    // shard's own; in the rare case that one needs more than that, the probe is repeated with four times as many
    for (size_t extra = 1;; extra *= 4) {
        const size_t cm = std::min(nch, c1 + extra);            // chunks [c0, cm) are mapped
        const uint64_t mapped_end = c1 == c0 ? f0 : (cm >= nch ? N : cstart[cm - 1] + clen[cm - 1]);
        { int rc = ensure_range(ctx, f0 ? f0 - 1 : 0, mapped_end); if (rc) return rc; }     // (the byte before the range: first byte of a chunk k >= 2)
        // ---- K1 ----
        uint32_t ncand = 0;
        {
            Phase ph(ctx, &ctx->st.ms_scan);
            CK(launch_scan_count(ctx->d_file, f0, f1, N, ctx->scan_flags, ctx->tile_counts.as<uint32_t>(), ctx->scan_masks.as<uint16_t>(), ctx->total.as<uint32_t>(), ctx->stream));
            CK(cudaMemcpyAsync(&ncand, ctx->total.p, 4, cudaMemcpyDeviceToHost, ctx->stream));
            CK(cudaStreamSynchronize(ctx->stream));
            ctx->st.kernel_launches += 2;
            cand.clear(); ctype.clear();
            if (ncand) {
                CK(ctx->cand.ensure((size_t)ncand * 4)); CK(ctx->ctype.ensure(ncand));
                CK(launch_scan_write(ctx->d_file, f0, f1, ctx->scan_masks.as<uint16_t>(), ctx->tile_counts.as<uint32_t>(), ctx->cand.as<uint32_t>(), ctx->ctype.as<uint8_t>(), ncand, ctx->stream));
                ctx->st.kernel_launches++;
                cand.resize(ncand); ctype.resize(ncand);
                CK(cudaMemcpyAsync(cand.data(), ctx->cand.p, (size_t)ncand * 4, cudaMemcpyDeviceToHost, ctx->stream));
                CK(cudaMemcpyAsync(ctype.data(), ctx->ctype.p, ncand, cudaMemcpyDeviceToHost, ctx->stream));
            }
            ph.stop();
            CK(cudaGetLastError());
            if (ctx->scan_flags & SPLIT_FLAGS) { k1cand = cand; k1type = ctype; }
        }
        // ---- the first position of every chunk k >= 2 holds file[start_k - 1] in the reference's buffer (see chunk_list): fix those up ----
        std::vector<uint8_t> special;    // per candidate: 1 = its first byte is file[off - 1]
        {
            const size_t k0 = std::max<size_t>(c0, 2);
            if (k0 < c1) {
                const size_t nb = c1 - k0;
                std::vector<uint8_t> edge(nb * 4, 0);       // file[p-1 .. p+2] of every boundary p = start_k
                if (ctx->h_file) { for (size_t i = 0; i < nb; i++) { const uint64_t p = cstart[k0 + i]; for (int b = 0; b < 4; b++) if (p - 1 + b < N) edge[4 * i + b] = ctx->h_file[p - 1 + b]; } }
                else if (S - 1 >= 4) {
                    CK(cudaMemcpy2DAsync(edge.data(), 4, ctx->d_file + cstart[k0] - 1, S - 1, 4, nb, cudaMemcpyDeviceToHost, ctx->stream));   // (reads stay inside the padded image)
                    CK(cudaStreamSynchronize(ctx->stream));
                } else {     // chunks of 2-4 bytes: rows would overlap, take the range as it is
                    const uint64_t lo = cstart[k0] - 1, hi = std::min<uint64_t>(N, cstart[c1 - 1] + 3);
                    std::vector<uint8_t> span(hi - lo);
                    CK(cudaMemcpyAsync(span.data(), ctx->d_file + lo, hi - lo, cudaMemcpyDeviceToHost, ctx->stream));
                    CK(cudaStreamSynchronize(ctx->stream));
                    for (size_t i = 0; i < nb; i++) for (int b2 = 0; b2 < 4; b2++) { const uint64_t q = cstart[k0 + i] - 1 + b2; if (q < hi) edge[4 * i + b2] = span[q - lo]; }
                }
                std::vector<uint32_t> c2; std::vector<uint8_t> t2, s2; c2.reserve(cand.size() + nb); t2.reserve(cand.size() + nb); s2.reserve(cand.size() + nb);
                size_t ci = 0;
                for (size_t i = 0; i < nb; i++) {
                    const uint64_t p = cstart[k0 + i];
                    while (ci < cand.size() && cand[ci] < p) { c2.push_back(cand[ci]); t2.push_back(ctype[ci]); s2.push_back(0); ci++; }
                    if (ci < cand.size() && cand[ci] == p) ci++;                       // what K1 saw there were the file's own bytes
                    const int ty = p + 1 < N ? zlib_header_type(edge[4 * i], edge[4 * i + 2], ctx->scan_flags) : -1;
                    if (ty >= 0) { c2.push_back((uint32_t)p); t2.push_back((uint8_t)ty); s2.push_back(1); }
                }
                while (ci < cand.size()) { c2.push_back(cand[ci]); t2.push_back(ctype[ci]); s2.push_back(0); ci++; }
                cand.swap(c2); ctype.swap(t2); special.swap(s2);
                ncand = (uint32_t)cand.size();
            }
            special.resize(ncand, 0);
        }
        ctx->st.n_candidates = ncand;
        // ---- K2 stage 1: every candidate inflates into a small slot of its own (plaintext + token map); its input ends at the end of
        // its chunk and then continues over the following chunks the way refillInput feeds them (main.cpp:207-217) ----
        jobs.assign(ncand, InflateJob{}); res.assign(ncand, InflateResult{}); cres.assign(ncand, InflateResult{});
        std::vector<uint8_t> capped(ncand, 0);
        auto chunk_of = [&](uint64_t f) { return (size_t)(f / (S - 1)); };
        for (uint32_t k = 0; k < ncand; k++) {
            uint64_t f = cand[k]; size_t c = chunk_of(f);
            uint64_t avail = cstart[c] + clen[c] - f;
            uint64_t vtot = avail + suffix[c + 1] - suffix[cm];      // the following chunks that are mapped
            capped[k] = cm < nch;
            jobs[k] = InflateJob{f, avail, vtot, (uint64_t)k * SLOT, Q, (uint64_t)k * SLOT + QS, (special[k] ? INFJ_FIRST_FROM_PREV : 0ull) | ((c == 0 ? 1ull : 0ull) << 8)};
        }
        // every candidate keeps its slot when they all fit in a quarter of the budget; a file that is mostly zlib headers
        // (tens of millions of candidates) is probed in batches that reuse the slots, and the few streams it really holds are
        // inflated once more afterwards
        const uint64_t per_batch = getenv("ATZ_SLOT_BATCH") ? (uint64_t)std::max(1, atoi(getenv("ATZ_SLOT_BATCH")))     // test hook
                                                            : std::max<uint64_t>(4096, std::max<uint64_t>(ctx->budget / 4, 1ull << 30) / SLOT);
        const bool resident = ncand <= per_batch;
        sc.resident = resident;
        if (ncand) {
            const uint64_t nslot = resident ? ncand : per_batch;
            CK(ctx->plain.ensure(nslot * SLOT + ATZ_PAD));
            for (uint64_t b0 = 0; b0 < ncand; b0 += nslot) {
                const uint64_t b1 = std::min<uint64_t>(ncand, b0 + nslot);
                CK(cudaMemsetAsync(ctx->plain.p, 0, (b1 - b0) * SLOT + ATZ_PAD, ctx->stream));
                if (resident) { int rc = run_inflate(ctx, ctx->d_file, jobs, res, cres, ctx->plain.as<uint8_t>(), S, &ctx->st.ms_inflate_probe); if (rc) return rc; }
                else {
                    std::vector<InflateJob> bj(jobs.begin() + b0, jobs.begin() + b1); std::vector<InflateResult> br, bc;
                    for (size_t i = 0; i < bj.size(); i++) { bj[i].out_off = (uint64_t)i * SLOT; bj[i].tmap_off = (uint64_t)i * SLOT + QS; }
                    int rc = run_inflate(ctx, ctx->d_file, bj, br, bc, ctx->plain.as<uint8_t>(), S, &ctx->st.ms_inflate_probe); if (rc) return rc;
                    std::copy(br.begin(), br.end(), res.begin() + b0); std::copy(bc.begin(), bc.end(), cres.begin() + b0);
                }
            }
        }
        // ---- K2 stage 2: the candidates that outgrew their slot, rerun with a region sized from the compressed bytes they can
        // cover (up to the next such candidate); a region that is still too small is enlarged and the job rerun ----
        sc.big_plain.assign(ncand, nullptr); sc.big_tmap.assign(ncand, nullptr);
        {
            std::vector<uint32_t> big; std::vector<uint64_t> cap;
            for (uint32_t k = 0; k < ncand; k++) if (res[k].status == INF_OUT_FULL || cres[k].status == INF_OUT_FULL) big.push_back(k);
            // region size: 5 x the compressed bytes the candidate can cover inside its chunk (text inflates ~3x; a false positive that
            // happens to survive its slot must not shrink a real stream's region, so the distance to the next candidate is NOT used);
            // if that is too much memory, fall back to the distance to the next such candidate and let the rerun loop fix what it cuts
            auto est_in = [&](uint32_t k) { return std::min<uint64_t>(std::min<uint64_t>(jobs[k].vtotal, jobs[k].avail + 65536), S + 65536); };   // a continuation rarely survives long
            uint64_t want = 0;
            for (uint32_t k : big) want += 2 * (align_up(std::max<uint64_t>(4 * Q, 5 * est_in(k)) + 16384, 256) + ATZ_PAD);
            const bool roomy = want <= ctx->budget / 4;
            for (size_t i = 0; i < big.size(); i++) {
                uint32_t k = big[i];
                uint64_t est = est_in(k);
                if (!roomy && i + 1 < big.size()) est = std::min<uint64_t>(est, (uint64_t)cand[big[i + 1]] - cand[k] + 256);
                cap.push_back(align_up(std::max<uint64_t>(4 * Q, 5 * est) + 16384, 256));
            }
            {   // longest first: the jobs run off a queue, one warp each
                std::vector<size_t> ord(big.size()); for (size_t i = 0; i < ord.size(); i++) ord[i] = i;
                std::stable_sort(ord.begin(), ord.end(), [&](size_t a, size_t b) { return cap[a] > cap[b]; });
                std::vector<uint32_t> b2(big.size()); std::vector<uint64_t> c2(big.size());
                for (size_t i = 0; i < ord.size(); i++) { b2[i] = big[ord[i]]; c2[i] = cap[ord[i]]; }
                big.swap(b2); cap.swap(c2);
            }
            int round = 0;
            while (!big.empty()) {
                uint64_t arena = 0; std::vector<InflateJob> bj(big.size()); std::vector<InflateResult> br, bc;
                for (size_t i = 0; i < big.size(); i++) {
                    InflateJob j = jobs[big[i]];
                    j.out_off = arena; j.out_cap = cap[i]; arena = align_up(arena + cap[i] + ATZ_PAD, 256);
                    j.tmap_off = arena; arena = align_up(arena + cap[i] + 64, 256);
                    bj[i] = j;
                }
                uint8_t *base;
                if (round == 0) { CK(ctx->plain2.ensure(arena + ATZ_PAD)); base = ctx->plain2.as<uint8_t>(); }
                else { void *q = nullptr; CK(cudaMalloc(&q, arena + ATZ_PAD)); ctx->plain_extra.push_back(q); base = (uint8_t *)q; }
                { int rc = run_inflate(ctx, ctx->d_file, bj, br, bc, base, S, &ctx->st.ms_inflate); if (rc) return rc; }
                if (getenv("ATZ_DEBUG_SCAN")) {
                    std::vector<size_t> o(big.size()); for (size_t i = 0; i < o.size(); i++) o[i] = i;
                    auto tout = [&](size_t i) { return std::max(br[i].total_out, bc[i].status >= 0 ? bc[i].total_out : 0); };
                    std::sort(o.begin(), o.end(), [&](size_t a, size_t b) { return tout(a) > tout(b); });
                    fprintf(stderr, "[scan] stage-2 round %d: %zu jobs\n", round, big.size());
                    for (size_t q = 0; q < std::min<size_t>(8, o.size()); q++) { size_t i = o[q];
                        fprintf(stderr, "   off %u avail %llu vtotal %llu cap %llu | probe st %d in %llu out %llu | cont st %d in %llu out %llu\n", cand[big[i]], (unsigned long long)jobs[big[i]].avail,
                                (unsigned long long)jobs[big[i]].vtotal, (unsigned long long)cap[i], br[i].status, (unsigned long long)br[i].total_in, (unsigned long long)br[i].total_out,
                                bc[i].status, (unsigned long long)bc[i].total_in, (unsigned long long)bc[i].total_out); }
                }
                std::vector<uint32_t> again; std::vector<uint64_t> cap2;
                for (size_t i = 0; i < big.size(); i++) {
                    uint32_t k = big[i];
                    if (br[i].status == INF_OUT_FULL || bc[i].status == INF_OUT_FULL) {
                        uint64_t lim = 1032 * jobs[k].vtotal + 65536;
                        if (cap[i] >= lim) { ctx->err = "inflate output exceeds the deflate expansion bound"; return ATZ_E_CUDA; }
                        again.push_back(k); cap2.push_back(std::min<uint64_t>(align_up(cap[i] * 6, 256), align_up(lim, 256)));
                    } else { res[k] = br[i]; cres[k] = bc[i]; sc.big_plain[k] = base + bj[i].out_off; sc.big_tmap[k] = base + bj[i].tmap_off; }
                }
                big.swap(again); cap.swap(cap2); round++;
            }
        }
        // a continuation that used up everything that was mapped without coming to an end needs more of the file
        bool starved = false;
        for (uint32_t k = 0; k < ncand && !starved; k++)
            starved = capped[k] && res[k].status == INF_NEED_INPUT && res[k].in_at_outcap > 16 && cres[k].status == INF_NEED_INPUT && cres[k].total_in >= jobs[k].vtotal;
        if (!starved) break;
        for (void *q : ctx->plain_extra) cudaFree(q);
        ctx->plain_extra.clear();
    }
    // ---- the records the accept logic can act on: everything else only ever makes it step to the next byte (main.cpp:229-241) ----
    std::vector<ProbeX> &mine = sc.px[shard];
    for (uint32_t k = 0; k < (uint32_t)cand.size(); k++) {
        if (res[k].in_at_outcap <= 16) continue;
        if (!(res[k].status == INF_END || res[k].total_in == jobs[k].avail)) continue;
        ProbeX x{}; x.off = cand[k]; x.avail = jobs[k].avail; x.local = k; x.type = ctype[k] | ((jobs[k].flags & INFJ_FIRST_FROM_PREV) ? 0x100u : 0u);
        x.p_status = res[k].status; x.p_in = res[k].total_in; x.p_out = res[k].total_out; x.p_cap = res[k].in_at_outcap; x.p_adler = res[k].adler;
        x.c_status = -1;
        if (res[k].status == INF_NEED_INPUT && cres[k].status >= 0) { x.c_status = cres[k].status; x.c_in = cres[k].total_in; x.c_out = cres[k].total_out; x.c_cap = cres[k].in_at_outcap; x.c_adler = cres[k].adler; }
        mine.push_back(x);
    }
    if (ctx->scan_flags & SPLIT_FLAGS) { int rc = probe_split_runs(ctx, k1cand, k1type); if (rc) return rc; }
    sc.have[shard] = 1; sc.probed = true;
    ctx->st.algo_bytes += f1 - f0;
    return ATZ_OK;
}

// the export: the exporting context's scan flags (8 bytes; the records were found with that header set), then the records; with
// ATZ_SCAN_PNG_IDAT or ATZ_SCAN_APNG_FDAT then the split streams (SPLIT_HEAD bytes each: off, C, U, adler, type, number of pieces; then
// the piece lengths) and the size of that part (8 bytes).  The type word of a stream split over fdAT chunks has SPLIT_FDAT set (an
// IDAT one's is the header type alone, as before fdAT runs existed).
#define SPLIT_HEAD 36
#define SPLIT_FDAT 0x10000u
int atz_probe_export(atz_ctx *ctx, void *buf, uint64_t cap, uint64_t *nbytes) {
    if (!ctx || !nbytes) return ATZ_E_ARG;
    if (!ctx->sc.probed) return ATZ_E_STATE;
    const std::vector<ProbeX> &v = ctx->sc.px[ctx->sc.shard];
    const uint64_t flags = ctx->scan_flags;
    std::vector<uint8_t> split;
    if (flags & SPLIT_FLAGS) {
        for (const SplitX &x : ctx->sc.split[ctx->sc.shard]) {
            uint8_t h[SPLIT_HEAD]; const uint32_t np = (uint32_t)x.pieces.size(), t = x.type | (x.frame == 16 ? SPLIT_FDAT : 0);
            memcpy(h, &x.off, 8); memcpy(h + 8, &x.c, 8); memcpy(h + 16, &x.u, 8); memcpy(h + 24, &x.adler, 4); memcpy(h + 28, &t, 4); memcpy(h + 32, &np, 4);
            split.insert(split.end(), h, h + SPLIT_HEAD);
            split.insert(split.end(), (const uint8_t *)x.pieces.data(), (const uint8_t *)(x.pieces.data() + np));
        }
        const uint64_t sb = split.size(); split.insert(split.end(), (const uint8_t *)&sb, (const uint8_t *)&sb + 8);
    }
    *nbytes = sizeof flags + v.size() * sizeof(ProbeX) + split.size();
    if (!buf || cap < *nbytes) return ATZ_E_SMALL;
    memcpy(buf, &flags, sizeof flags);
    if (!v.empty()) memcpy((uint8_t *)buf + sizeof flags, v.data(), v.size() * sizeof(ProbeX));
    if (!split.empty()) memcpy((uint8_t *)buf + sizeof flags + v.size() * sizeof(ProbeX), split.data(), split.size());
    return ATZ_OK;
}
int atz_probe_import(atz_ctx *ctx, uint32_t shard, const void *buf, uint64_t nbytes) {
    uint64_t flags = 0, split_bytes = 0;
    if (!ctx || !buf || nbytes < sizeof flags) return ATZ_E_ARG;
    const uint8_t *b = (const uint8_t *)buf;
    memcpy(&flags, b, sizeof flags);
    if (flags & SPLIT_FLAGS) {     // the split streams and their size behind the probe records
        if (nbytes < 2 * sizeof flags) return ATZ_E_ARG;
        memcpy(&split_bytes, b + nbytes - 8, 8);
        if (split_bytes > nbytes - 16) return ATZ_E_ARG;
        split_bytes += 8;
    }
    if ((nbytes - sizeof flags - split_bytes) % sizeof(ProbeX)) return ATZ_E_ARG;
    if (!ctx->sc.probed) return ATZ_E_STATE;
    if (shard >= ctx->sc.nshards || shard == ctx->sc.shard) return ATZ_E_ARG;
    if (flags != ctx->scan_flags) { ctx->set_err("atz_probe_import: the shard scanned with other scan flags (atz_ctx_set_scan_flags)"); return ATZ_E_STATE; }
    nbytes -= sizeof flags + split_bytes;
    std::vector<ProbeX> &v = ctx->sc.px[shard];
    v.resize(nbytes / sizeof(ProbeX));
    if (nbytes) memcpy(v.data(), b + sizeof flags, nbytes);
    for (size_t i = 0; i < v.size(); i++) if (v[i].off >= ctx->n || (i && v[i].off <= v[i - 1].off)) return ATZ_E_ARG;
    std::vector<SplitX> &sv = ctx->sc.split[shard]; sv.clear();
    for (const uint8_t *q = b + sizeof flags + nbytes, *e = q + (split_bytes ? split_bytes - 8 : 0); q < e;) {
        if (e - q < SPLIT_HEAD) return ATZ_E_ARG;
        SplitX x; uint32_t np = 0, t = 0;
        memcpy(&x.off, q, 8); memcpy(&x.c, q + 8, 8); memcpy(&x.u, q + 16, 8); memcpy(&x.adler, q + 24, 4); memcpy(&t, q + 28, 4); memcpy(&np, q + 32, 4);
        q += SPLIT_HEAD;
        const bool fdat = t & SPLIT_FDAT;    // the kind must be one the scan flags enable
        x.type = t & ~SPLIT_FDAT; x.frame = fdat ? 16 : 12;
        if (!(flags & (fdat ? ATZ_SCAN_APNG_FDAT : ATZ_SCAN_PNG_IDAT))) return ATZ_E_ARG;
        if (np < 2 || (uint64_t)(e - q) / 4 < np) return ATZ_E_ARG;
        x.pieces.resize(np); memcpy(x.pieces.data(), q, 4ull * np); q += 4ull * np;
        uint64_t sum = 0; for (uint32_t l : x.pieces) sum += l;
        if (sum != x.c || x.type >= ATZ_NTYPES || x.off >= ctx->n || x.span() > ctx->n - x.off || (!sv.empty() && x.off <= sv.back().off)) return ATZ_E_ARG;
        sv.push_back(std::move(x));
    }
    ctx->sc.have[shard] = 1;
    return ATZ_OK;
}

int atz_scan_finish(atz_ctx *ctx, uint64_t *n_streams) {
    if (!ctx) return ATZ_E_ARG;
    ScanState &sc = ctx->sc;
    if (!sc.probed) return ATZ_E_STATE;
    for (uint8_t h : sc.have) if (!h) { ctx->set_err("atz_scan_finish: the probe records of a shard are missing (atz_probe_import)"); return ATZ_E_STATE; }
    cudaSetDevice(ctx->device);
    const uint64_t N = ctx->n, S = sc.S;
    std::vector<uint64_t> cstart, clen;
    chunk_list(N, S, cstart, clen);
    // ---- the sequential accept logic, chunk by chunk, over the records of all shards (file order = shard order) ----
    std::vector<const ProbeX *> all; std::vector<uint32_t> src;
    for (uint32_t g = 0; g < sc.nshards; g++) for (const ProbeX &x : sc.px[g]) { all.push_back(&x); src.push_back(g); }
    const uint32_t nx = (uint32_t)all.size();
    std::vector<Acc> acc;
    {
        std::vector<uint32_t> xc(nx); std::vector<ProbeRec> pr(nx), cr; std::vector<uint64_t> avail(nx); std::vector<int32_t> cont_of(nx, -1);
        for (uint32_t k = 0; k < nx; k++) {
            const ProbeX &x = *all[k];
            xc[k] = (uint32_t)x.off; pr[k] = ProbeRec{x.p_status, x.p_in, x.p_out, x.p_cap}; avail[k] = x.avail;
            if (x.c_status >= 0) { cont_of[k] = (int32_t)cr.size(); cr.push_back(ProbeRec{x.c_status, x.c_in, x.c_out, x.c_cap}); }
        }
        scan_fold(cstart, clen, xc.data(), nx, pr.data(), avail.data(), cont_of.data(), cr.data(), acc);
    }
    // ---- ATZ_SCAN_PNG_IDAT / ATZ_SCAN_APNG_FDAT, after the fold and the same on every context: a split stream (IDAT and fdAT runs in one
    // list, file order) is dropped if an accepted stream
    // or a split stream kept before it overlaps its span without lying inside it; otherwise it takes the place of the accepted streams
    // inside its span (accidents of inflating compressed bytes) ----
    struct SplitRef { const SplitX *x; uint32_t src, local; };
    std::vector<SplitRef> spl; std::vector<int32_t> split_of;     // split_of[s]: stream s is spl[split_of[s]] (-1: an accepted stream of the fold)
    for (uint32_t g = 0; g < sc.nshards; g++) for (uint32_t i = 0; i < (uint32_t)sc.split[g].size(); i++) spl.push_back(SplitRef{&sc.split[g][i], g, i});
    if (!spl.empty()) {
        std::vector<uint64_t> pmax(acc.size());   // largest end of acc[0 .. j]
        for (size_t j = 0; j < acc.size(); j++) pmax[j] = std::max(j ? pmax[j - 1] : 0, acc[j].off + acc[j].tin);
        std::vector<uint8_t> gone(acc.size(), 0); std::vector<uint32_t> kept; uint64_t last = 0;
        for (uint32_t q = 0; q < (uint32_t)spl.size(); q++) {
            const uint64_t a = spl[q].x->off, b = a + spl[q].x->span();
            if (a < last) continue;
            const size_t j0 = std::lower_bound(acc.begin(), acc.end(), a, [](const Acc &u, uint64_t v) { return u.off < v; }) - acc.begin();
            if (j0 && pmax[j0 - 1] > a) continue;
            size_t j1 = j0; bool inside = true;
            for (; j1 < acc.size() && acc[j1].off < b; j1++) if (acc[j1].off + acc[j1].tin > b) { inside = false; break; }
            if (!inside) continue;
            for (size_t j = j0; j < j1; j++) gone[j] = 1;
            kept.push_back(q); last = b;
        }
        std::vector<Acc> m; size_t k = 0;
        for (size_t j = 0; j <= acc.size(); j++) {
            for (; k < kept.size() && (j == acc.size() || spl[kept[k]].x->off < acc[j].off); k++) {
                const SplitX &x = *spl[kept[k]].x;
                m.push_back(Acc{x.off, x.c, x.u, kept[k], false}); split_of.push_back((int32_t)kept[k]);
            }
            if (j < acc.size() && !gone[j]) { m.push_back(acc[j]); split_of.push_back(-1); }
        }
        acc.swap(m);
    }
    split_of.resize(acc.size(), -1);
    // ---- accepted streams; the ones this shard owns get their plaintext (already resident where this context probed them) ----
    const size_t ns = acc.size();
    std::vector<uint64_t> ulen(ns); std::vector<uint32_t> owner(ns, 0);
    for (size_t s = 0; s < ns; s++) ulen[s] = acc[s].tout;
    std::vector<uint32_t> probed_by(ns);
    for (size_t s = 0; s < ns; s++) probed_by[s] = split_of[s] >= 0 ? spl[split_of[s]].src : src[acc[s].cand];
    stream_partition(ulen.data(), probed_by.data(), (uint32_t)ns, sc.nshards, owner.data());
    ctx->streams.assign(ns, StreamRec{});
    std::vector<size_t> recheck, far_runs; uint64_t far_bytes = 0;
    for (size_t s = 0; s < ns; s++) {
        if (acc[s].tout >= 0xffffff00ull || acc[s].tin >= 0xffffff00ull) return ATZ_E_TOO_LARGE;
        StreamRec &r = ctx->streams[s];
        r.s = atz_stream{}; r.s.offset = acc[s].off; r.s.streamLength = acc[s].tin; r.s.inflatedLength = acc[s].tout;
        r.s.clevel = 9; r.s.window = 15; r.s.memlevel = 9; r.s.firstDiffByte = -1;
        if (split_of[s] >= 0) {     // a split stream: its bytes are resident where it was probed; another owner puts its pieces together and inflates them again
            const SplitRef &q = spl[split_of[s]];
            r.s.offsetType = (int32_t)q.x->type; r.owner = owner[s]; r.adler = q.x->adler; r.pieces = q.x->pieces; r.frame = q.x->frame;
            if (r.owner != sc.shard) continue;
            if (q.src == sc.shard) { const SplitDev &d = sc.split_dev[q.local]; r.d_comp = d.comp; r.d_plain = d.plain; r.d_tmap = d.tmap; }
            else { far_runs.push_back(s); recheck.push_back(s); }
            ctx->st.algo_bytes += acc[s].tin + acc[s].tout;
            continue;
        }
        const ProbeX &x = *all[acc[s].cand];
        r.s.offsetType = (int32_t)(x.type & 0xff); r.owner = owner[s];
        r.adler = acc[s].via_cont ? x.c_adler : x.p_adler;
        if (r.owner != sc.shard) continue;
        const bool here = src[acc[s].cand] == sc.shard;
        const uint32_t k = x.local;
        if (here && !acc[s].via_cont && !(x.type & 0x100u) && (sc.big_plain[k] || sc.resident)) {      // (a stream probed with a foreign first byte is inflated again from the real bytes, like one accepted across a boundary)
            if (sc.big_plain[k]) { r.d_plain = sc.big_plain[k]; r.d_tmap = sc.big_tmap[k]; }
            else { r.d_plain = ctx->plain.as<uint8_t>() + (uint64_t)k * sc.SLOT; r.d_tmap = r.d_plain + sc.QS; }
        } else recheck.push_back(s);   // no resident plaintext (probed elsewhere, across a chunk boundary, or in reused slots): inflate the real file bytes
        if (acc[s].off >= ctx->r0 && acc[s].off + acc[s].tin <= ctx->r1) r.d_comp = ctx->d_file + acc[s].off;
        else far_bytes += align_up(acc[s].tin + ATZ_PAD, 256);
        ctx->st.algo_bytes += acc[s].tin + acc[s].tout;
    }
    if (!far_runs.empty()) {   // (before the staging below, which takes every owned stream that has no compressed bytes yet)
        std::vector<RunBytes> rb;
        for (size_t s : far_runs) { const StreamRec &r = ctx->streams[s]; rb.push_back(RunBytes{r.s.offset, r.pieces.data(), r.pieces.size(), r.s.streamLength, r.frame}); }
        uint8_t *base = nullptr; std::vector<uint64_t> at;
        { int rc = dechunk(ctx, rb, base, at); if (rc) return rc; }
        for (size_t i = 0; i < far_runs.size(); i++) ctx->streams[far_runs[i]].d_comp = base + at[i];
    }
    if (far_bytes) {   // compressed bytes of owned streams outside the mapped range: staged (one pinned-free gather on the host side, one copy)
        if (!ctx->h_file) { ctx->set_err("owned stream outside the resident file range"); return ATZ_E_STATE; }
        CK(ctx->comp_extra.ensure(far_bytes + ATZ_PAD));
        std::vector<uint8_t> stage(far_bytes, 0); uint64_t o = 0;
        for (size_t s = 0; s < ns; s++) {
            StreamRec &r = ctx->streams[s];
            if (r.owner != sc.shard || r.d_comp) continue;
            memcpy(stage.data() + o, ctx->h_file + r.s.offset, r.s.streamLength);
            r.d_comp = ctx->comp_extra.as<uint8_t>() + o; o += align_up(r.s.streamLength + ATZ_PAD, 256);
        }
        Phase ph(ctx, &ctx->st.ms_h2d);
        CK(cudaMemcpyAsync(ctx->comp_extra.p, stage.data(), far_bytes, cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaMemsetAsync(ctx->comp_extra.as<uint8_t>() + far_bytes, 0, ATZ_PAD, ctx->stream));
        ph.stop();
    }
    if (!recheck.empty()) {
        // a stream accepted across a chunk boundary saw a duplicated byte; phase 3 inflates the real file bytes (doInflate, main.cpp:441)
        // and the reference aborts when that fails (main.cpp:450-453)
        uint64_t arena = 0; std::vector<InflateJob> vj(recheck.size()); std::vector<InflateResult> vr, vc;
        const uint8_t *base = nullptr;    // job offsets are relative to the lowest compressed-bytes address of the group
        for (size_t i : recheck) { const uint8_t *c = ctx->streams[i].d_comp; if (!base || c < base) base = c; }
        {   // longest first
            std::stable_sort(recheck.begin(), recheck.end(), [&](size_t a, size_t b) { return acc[a].tout > acc[b].tout; });
        }
        for (size_t i = 0; i < recheck.size(); i++) {
            const Acc &a = acc[recheck[i]]; uint64_t in = std::min<uint64_t>(a.tin, N - a.off);
            vj[i] = InflateJob{(uint64_t)(ctx->streams[recheck[i]].d_comp - base), in, in, arena, a.tout, ~0ull, 0}; arena = align_up(arena + a.tout + ATZ_PAD, 256);
            vj[i].tmap_off = arena; arena = align_up(arena + a.tout + 64, 256);
        }
        void *q = nullptr; CK(cudaMalloc(&q, arena + ATZ_PAD)); ctx->plain_extra.push_back(q);
        CK(cudaMemsetAsync(q, 0, arena + ATZ_PAD, ctx->stream));
        { int rc = run_inflate(ctx, base, vj, vr, vc, (uint8_t *)q, S, &ctx->st.ms_inflate); if (rc) return rc; }
        for (size_t i = 0; i < recheck.size(); i++) {
            if (vr[i].status != INF_END || vr[i].total_out != acc[recheck[i]].tout) { ctx->err = "inflate() failed on an accepted stream (reference would abort, main.cpp:451)"; return ATZ_E_DATA; }
            StreamRec &r = ctx->streams[recheck[i]];
            if (!r.pieces.empty() && (vr[i].total_in != r.s.streamLength || vr[i].adler != r.adler)) { ctx->set_err("a split stream inflates differently on its owner than where it was probed"); return ATZ_E_DATA; }
            r.d_plain = (uint8_t *)q + vj[i].out_off; r.d_tmap = (uint8_t *)q + vj[i].tmap_off; r.adler = vr[i].adler;
        }
    }
    ctx->st.n_streams = ns;
    if (n_streams) *n_streams = ns;
    ctx->state = 2;
    return ATZ_OK;
}

int atz_scan(atz_ctx *ctx, uint64_t chunksize, uint64_t *n_streams) {
    int rc = atz_scan_shard(ctx, chunksize, 0, 1);
    return rc ? rc : atz_scan_finish(ctx, n_streams);
}

// ---------------------------------------------------------------------------------------------
int atz_search(atz_ctx *ctx, const atz_options *opt) { return atz_search_shard(ctx, opt, 0, 1); }

// counters of a lane go into the context's (sums; the lane's are cleared)
static void merge_lane_stats(atz_ctx *ctx, Lane &L) {
    const atz_stats a = L.st; L.st = atz_stats{};
    ctx->st.ms_chains += a.ms_chains; ctx->st.ms_rows += a.ms_rows; ctx->st.ms_trials += a.ms_trials; ctx->st.ms_diff += a.ms_diff;
    ctx->st.kernel_launches += a.kernel_launches; ctx->st.n_trial_kernels += a.n_trial_kernels; ctx->st.gpu_trials += a.gpu_trials;
    ctx->st.ref_trials += a.ref_trials; ctx->st.trial_algo_bytes += a.trial_algo_bytes;
    ctx->st.ms_trials_max_kernel = std::max(ctx->st.ms_trials_max_kernel, a.ms_trials_max_kernel);
}

// The search of one lane: the streams `sidx` (indices into R: ctx->streams, or ctx->nested), in batches whose chain structures fit the lane's budget.
static int search_lane(atz_ctx *ctx, Lane &L, const atz_options *opt, const TrialOpts &topts, std::vector<StreamRec> &R, const std::vector<uint32_t> &sidx,
                       const std::vector<Params> *seq_class, const std::vector<Params> *seq_brute, const std::vector<Params> *seq_strat) {
    cudaSetDevice(ctx->device);
    const size_t ns = sidx.size();
    std::vector<PlainView> views(ns);
    for (size_t j = 0; j < ns; j++) {
        const StreamRec &r = R[sidx[j]];
        views[j] = PlainView{r.d_plain, (uint32_t)r.s.inflatedLength, r.d_comp, (uint32_t)r.s.streamLength, r.adler, r.d_tmap};
    }
    auto S = [&](size_t j) -> atz_stream & { return R[sidx[j]].s; };
    const size_t slots_share = std::max<size_t>(64, (size_t)trial_slots(ctx) / (size_t)std::max(1, ctx->nlanes_last));   // speculation depth as if the lanes shared one launch
    CK(L.queue.ensure(64));
    struct Prog { const std::vector<Params> *sq = nullptr; size_t next = 0; int phase = 0; bool done = false; };   // phase 0 = header class, 1 = brute window, 2 = other strategies (extension)
    std::vector<Prog> prog(ns);
    for (size_t j = 0; j < ns; j++) prog[j].sq = &seq_class[S(j).offsetType];
    // one batch: the streams js (indices into sidx) from where they are in their sequences until they are done or deferred
    // chain_limit: bytes of bucket lists the batch may build before it starts deferring streams (<= the arena)
    auto run_batch = [&](const std::vector<size_t> &js, uint64_t chain_bytes_wanted, uint64_t chain_limit) -> int {
        const size_t nb = js.size();
        { int rc = chain_arena_for(ctx, L, chain_bytes_wanted); if (rc) return rc; }
        chain_limit = std::min<uint64_t>(chain_limit, L.chains.cap);
        // row tables of up to 12 (hash size, level class) keys per stream plus as much again for the transient resolved tables
        { uint64_t rw = 0; for (size_t j : js) rw += 24 * (32 * (S(j).inflatedLength + 32) + 256); rec_arena_for(ctx, L, rw); }
        ChainState cs; cs.init(views.size());
        // The winner fold of one stream over the final results of `count` consecutive candidates (main.cpp:685-700), and what comes
        // next for it: more of its sequence, the --brute-window grid (main.cpp:590-601), or nothing.
        auto fold_span = [&](size_t j, const TrialResult *r, size_t count) {     // j: index into js
            Prog &p = prog[js[j]];
            atz_stream &st = S(js[j]);
            bool full = false; size_t used = 0;
            for (size_t t = 0; t < count && !full; t++) {
                const Params &pr = (*p.sq)[p.next + t]; used++;
                if (p.phase < 2) L.st.ref_trials++;
                uint64_t cmp = r[t].status == TR_BAILED ? std::min<uint64_t>(opt->shortcutLength, r[t].out_len) : std::min<uint64_t>(r[t].out_len, st.streamLength);
                L.st.trial_algo_bytes += r[t].in_consumed + cmp;
                if (r[t].status == TR_COMPARED && (uint64_t)r[t].ident > st.identBytes) {
                    st.identBytes = r[t].ident; st.clevel = (uint8_t)(pr.c | (pr.s << 4)); st.window = pr.w; st.memlevel = pr.m;
                    full = (r[t].ident == st.streamLength) || ((uint64_t)r[t].ident + opt->mismatchTol >= st.streamLength);
                }
            }
            p.next += used;
            if (full || p.next >= p.sq->size()) {
                const bool matched = st.identBytes == st.streamLength || st.identBytes + opt->mismatchTol >= st.streamLength;
                if (p.phase == 0 && opt->bruteforceWindow && (st.streamLength - st.identBytes) >= opt->mismatchTol) {   // main.cpp:590
                    p.phase = 1; p.next = 0; p.sq = &seq_brute[st.offsetType];
                    // window 11-14: a fullmatch in the lower range returns before the upper one (main.cpp:597); both ranges stop at the first fullmatch
                } else if (p.phase < 2 && (opt->flags & ATZ_F_STRATEGIES) && !matched) {
                    p.phase = 2; p.next = 0; p.sq = &seq_strat[st.offsetType];
                } else p.done = true;
            }
        };
        // Waves.  Phase A: every candidate of the wave up to the --shortcut-len prefix test (what testDeflateParams' first deflate()
        // call decides, main.cpp:632-653).  Phase B: the candidates that passed it, in full, with whole-stream rows and resolved tables.
        // A phase-B launch is a few long trials (its length is that of its longest one), so it runs in the BACKGROUND on the side
        // stream while the streams that have nothing in it go through their next wave; a stream with a candidate in phase B is parked
        // (its fold needs that result before anything later) and rejoins when the launch has been collected.  Results never depend on
        // this (trials are independent, the fold order per stream is kept); ATZ_BG_B=0 runs phase B in the foreground (test hook).
        const bool bg_on = !(getenv("ATZ_BG_B") && atoi(getenv("ATZ_BG_B")) == 0);
        struct Park { size_t j; std::vector<TrialResult> res; std::vector<std::pair<size_t, size_t>> fix; };   // fix: (index in res, index in the pending launch)
        std::vector<Park> parked; std::vector<uint8_t> is_parked(nb, 0), deferred(nb, 0);
        Launched bln; std::vector<TrialReq> breqs; bool b_pending = false;
        int wave = 0;
        for (;;) {
            size_t active = 0; for (size_t j = 0; j < nb; j++) if (!prog[js[j]].done && !is_parked[j] && !deferred[j]) active++;
            if (!active && !b_pending) break;
            uint64_t planned = cs.chain_used;     // bucket-list bytes in use once this wave's new hash sizes are built
            std::vector<TrialReq> reqs; std::vector<std::pair<size_t, size_t>> span(nb, {0, 0});   // first request, count
            if (active) {
                size_t k0 = std::max<size_t>(1, slots_share / active);
                const size_t growth = getenv("ATZ_WAVE_GROWTH") ? (size_t)std::max(2, atoi(getenv("ATZ_WAVE_GROWTH"))) : 4;   // (tuning hook)
                for (int w = 0; w < wave && k0 < 1024; w++) k0 *= growth;
                for (size_t j = 0; j < nb; j++) {
                    Prog &p = prog[js[j]]; span[j] = {reqs.size(), 0};
                    if (p.done || is_parked[j] || deferred[j]) continue;
                    const std::vector<Params> &seq = *p.sq;
                    const atz_stream &sj = S(js[j]);
                    // (a stream that comes back from a deferral is past its first wave: it takes the larger step of a second wave)
                    size_t k = p.phase >= 1 ? seq.size() - p.next : std::min(p.next > 0 && wave == 0 ? k0 * growth : k0, seq.size() - p.next);
                    if (p.next == 0 && p.phase == 0) {
                        // first wave: the leading candidates that share one memLevel (one set of chains and rows serves them all); the
                        // reference's order puts zlib's default memLevel 8 first, where streams made by zlib resolve (SURVEY.md A.2)
                        size_t run = 1; while (run < 4 && p.next + run < seq.size() && seq[p.next + run].m == seq[p.next].m) run++;
                        k = std::max(std::min(k, seq.size() - p.next), run);
                        if (active * 2 > slots_share) k = run;
                    }
                    {   // room for the bucket lists these candidates need?  If not, the stream waits for a later batch (never the batch's first)
                        uint32_t newm = 0;
                        for (size_t t = 0; t < k; t++) { const Params &q = seq[p.next + t]; if (needs_chain(q) && !cs.chain((uint32_t)js[j], q.m).list) newm |= 1u << q.m; }
                        const uint64_t need = (uint64_t)__builtin_popcount(newm) * chain_bytes(sj.inflatedLength);
                        if (need && planned + need > chain_limit && nb > 1 && (planned > 0 || j > 0)) { deferred[j] = 1; continue; }
                        planned += need;
                    }
                    for (size_t t = 0; t < k; t++) {
                        TrialReq rq{(uint32_t)js[j], seq[p.next + t], 0, nullptr, 0};
                        // row tables: the whole stream where the trial is likely to run to the end (zlib's default memLevel, or a stream
                        // hardly longer than its first block), the first block otherwise (a trial that outlives its table walks the chains);
                        // deflate_fast rows only where the header's FLEVEL makes that level plausible (Z/deflate.c:741-748)
                        const int cls = sj.offsetType % 4;
                        // a stream hardly longer than the candidate's first block is simply run to the end
                        // (and so is one whose compressed form is no longer than --shortcut-len: testDeflateParams has no prefix test then, main.cpp:632)
                        rq.phase1 = (sj.inflatedLength > 4ull * (64u << rq.prm.m) + 4096 && sj.streamLength > opt->shortcutLength) ? 1 : 0;
                        // rows at every position for the candidates that are unlikely to reproduce the original (later waves, the brute grid):
                        // their parse looks where the original's did not
                        if (!needs_chain(rq.prm)) { }
                        else if (rq.prm.c >= 4) { rq.want_rec = rq.phase1 ? 1 : 2; rq.want_res = 1; rq.reserve_whole = p.phase == 0 && p.next == 0; rq.all_rows = p.phase >= 1 || p.next > 0; }
                        else if (rq.prm.c >= 1) rq.want_rec = (p.phase == 0 && ((cls == 0 && rq.prm.c == 1) || (cls == 1 && rq.prm.c >= 2))) ? 2 : 0;
                        reqs.push_back(rq);
                    }
                    span[j].second = k;
                }
            }
            std::vector<TrialResult> tr;
            { int rc = run_trials(ctx, L, views, reqs, topts, cs, tr, true); if (rc) return rc; }
            // the background launch of the wave before has had this wave's time to finish: its streams are folded and rejoin
            if (b_pending) {
                std::vector<TrialResult> trb(breqs.size());
                { int rc = collect_trials(ctx, L, bln, trb); if (rc) return rc; }
                b_pending = false;
                for (Park &pk : parked) {
                    for (auto &f : pk.fix) pk.res[f.first] = trb[f.second];
                    is_parked[pk.j] = 0;
                    fold_span(pk.j, pk.res.data(), pk.res.size());
                }
                parked.clear(); breqs.clear();
            }
            // this wave: streams without a prefix survivor are folded now, the others wait for phase B
            for (size_t j = 0; j < nb; j++) {
                if (!span[j].second) continue;
                const TrialResult *r = tr.data() + span[j].first;
                Park pk; pk.j = j;
                for (size_t t = 0; t < span[j].second; t++) if (r[t].status == TR_PASSED) {
                    TrialReq rq = reqs[span[j].first + t];
                    rq.phase1 = 0;
                    if (rq.prm.c >= 4 && needs_chain(rq.prm)) { rq.want_rec = 2; rq.want_res = 1; }
                    pk.fix.push_back({t, breqs.size()}); breqs.push_back(rq);
                }
                if (pk.fix.empty()) { fold_span(j, r, span[j].second); continue; }
                pk.res.assign(r, r + span[j].second);
                is_parked[j] = 1; parked.push_back(std::move(pk));
            }
            if (!breqs.empty()) {
                std::vector<TrialResult> dummy;
                if (bg_on) {
                    { int rc = run_trials(ctx, L, views, breqs, topts, cs, dummy, false, &bln); if (rc) return rc; }   // long trials: the full-register build
                    b_pending = true;
                } else {
                    { int rc = run_trials(ctx, L, views, breqs, topts, cs, dummy, false); if (rc) return rc; }
                    for (Park &pk : parked) {
                        for (auto &f : pk.fix) pk.res[f.first] = dummy[f.second];
                        is_parked[pk.j] = 0;
                        fold_span(pk.j, pk.res.data(), pk.res.size());
                    }
                    parked.clear(); breqs.clear();
                }
            }
            wave++;
        }
        // ---- recomp decision + diff lists of imperfect winners (main.cpp:454-456, 699-715) ----
        std::vector<size_t> need;
        uint64_t tmp_bytes = 0;
        for (size_t j : js) {
            if (!prog[j].done) continue;       // (deferred to a later batch)
            atz_stream &st = S(j);
            st.recomp = ((st.streamLength - st.identBytes) <= opt->recompTresh) && st.identBytes > 0;
            if (st.recomp && st.identBytes < st.streamLength) { need.push_back(j); tmp_bytes += align_up(st.streamLength + opt->sizediffTresh + 64, 256); }
        }
        if (!need.empty()) {
            CK(L.tmp_out.ensure(tmp_bytes)); CK(cudaMemsetAsync(L.tmp_out.p, 0, tmp_bytes, L.stream));
            std::vector<TrialReq> reqs; uint64_t o = 0; std::vector<uint64_t> offs;
            for (size_t j : need) {
                atz_stream &st = S(j); uint32_t cap = (uint32_t)align_up(st.streamLength + opt->sizediffTresh + 64, 256);
                { TrialReq rq{(uint32_t)j, Params{(uint8_t)(st.clevel & 15), st.window, st.memlevel, (uint8_t)(st.clevel >> 4)}, 1, L.tmp_out.as<uint8_t>() + o, cap};
                  if (needs_chain(rq.prm)) { rq.want_rec = 2; rq.want_res = 1; } reqs.push_back(rq); } offs.push_back(o); o += cap;
            }
            std::vector<TrialResult> tr; TrialOpts so = make_opts(nullptr, false);
            uint64_t before = L.st.gpu_trials;
            { int rc = run_trials(ctx, L, views, reqs, so, cs, tr); if (rc) return rc; }
            L.st.gpu_trials = before + reqs.size();
            uint64_t dcap = 0; for (size_t j : need) dcap += S(j).streamLength - S(j).identBytes + 1;
            CK(L.tmp_pos.ensure(dcap * 4)); CK(L.tmp_val.ensure(dcap)); CK(L.tmp_cnt.ensure(need.size() * 4)); CK(L.djobs.ensure(need.size() * sizeof(DiffJob)));
            std::vector<DiffJob> dj; uint64_t dpos = 0; std::vector<uint64_t> dstart;
            for (size_t q = 0; q < need.size(); q++) {
                atz_stream &st = S(need[q]); uint32_t cap = (uint32_t)(st.streamLength - st.identBytes + 1);
                dj.push_back(DiffJob{L.tmp_out.as<uint8_t>() + offs[q], R[sidx[need[q]]].d_comp, tr[q].out_len, (uint32_t)st.streamLength,
                                     L.tmp_pos.as<uint32_t>() + dpos, L.tmp_val.as<uint8_t>() + dpos, cap, L.tmp_cnt.as<uint32_t>() + q});
                dstart.push_back(dpos); dpos += cap;
            }
            CK(cudaMemcpyAsync(L.djobs.p, dj.data(), dj.size() * sizeof(DiffJob), cudaMemcpyHostToDevice, L.stream));
            {
                Phase ph(L, &L.st.ms_diff, "diff");
                CK(launch_diff(L.djobs.as<DiffJob>(), (uint32_t)dj.size(), L.stream));
                ph.stop(); L.st.kernel_launches++;
            }
            std::vector<uint32_t> hpos(dcap), hcnt(need.size()); std::vector<uint8_t> hval(dcap);
            CK(cudaMemcpyAsync(hpos.data(), L.tmp_pos.p, dcap * 4, cudaMemcpyDeviceToHost, L.stream));
            CK(cudaMemcpyAsync(hval.data(), L.tmp_val.p, dcap, cudaMemcpyDeviceToHost, L.stream));
            CK(cudaMemcpyAsync(hcnt.data(), L.tmp_cnt.p, need.size() * 4, cudaMemcpyDeviceToHost, L.stream));
            CK(cudaStreamSynchronize(L.stream));
            for (size_t q = 0; q < need.size(); q++) {
                StreamRec &r = R[sidx[need[q]]]; uint32_t nd = hcnt[q];
                if (nd != r.s.streamLength - r.s.identBytes) { ctx->set_err("diff pass disagrees with the trial's ident count"); return ATZ_E_CUDA; }
                r.s.firstDiffByte = hpos[dstart[q]]; r.s.ndiff = nd;
                r.diff_off.resize(nd); r.diff_val.resize(nd);
                for (uint32_t i = 0; i < nd; i++) {   // deltaEncode, main.cpp:757-763
                    r.diff_off[i] = i == 0 ? 0 : (uint64_t)hpos[dstart[q] + i] - hpos[dstart[q] + i - 1];
                    r.diff_val[i] = hval[dstart[q] + i];
                }
            }
        }
        return ATZ_OK;
    };
    // Batches.  A stream needs one set of bucket lists if it resolves in its first wave and nine if it goes through its whole
    // sequence; which, is not known in advance.  Sizing every batch for nine sets per stream (round 1) made the 1 GB corpus seven
    // batches, each with its own waves and their tails.  Now a batch is sized for `kSets` sets per stream (nine for a stream that has
    // been deferred before), and a stream whose next candidates need lists the arena has no room for any more is DEFERRED: it keeps
    // its place in its sequence and goes into a later batch.  Results do not depend on the batching (ATZ_BATCH_SETS: test hook).
    {
        const int sets_env = getenv("ATZ_BATCH_SETS") ? std::max(1, atoi(getenv("ATZ_BATCH_SETS"))) : 0;
        const uint64_t kSets = sets_env ? (uint64_t)sets_env : 3;
        std::vector<uint8_t> hard(ns, 0);
        std::vector<size_t> pending(ns); for (size_t j = 0; j < ns; j++) pending[j] = j;
        size_t rounds = 0;
        while (!pending.empty()) {
            uint64_t worst = 0; size_t i1 = 0;
            while (i1 < pending.size()) {
                const uint64_t add = (hard[pending[i1]] ? 9 : kSets) * chain_bytes(S(pending[i1]).inflatedLength);
                if (i1 > 0 && worst + add > L.budget / 2) break;
                worst += add; i1++;
            }
            std::vector<size_t> js(pending.begin(), pending.begin() + i1);
            // Who is in the batch is decided by the estimate; how much of the arena the batch may fill before it defers, by the size of
            // the job.  A small container (estimate up to a quarter of the budget) runs as one batch with room for nine sets for
            // everyone: nothing is deferred (128 MB mixed corpus: 682 ms per step against 859 when streams are deferred).  A large one
            // defers on purpose: a batch builds no more than its estimate, so the streams that go through their whole sequences leave
            // every batch and meet in the last ones - the long waves and the --brute-window launch happen once for the container, not
            // once per batch (1 GB: 4,764 against 5,456 ms; 512 MB is between the regimes and did not gain: DESIGN.md section 8).  The limit is explicit because the arena
            // itself only ever grows (a later batch of deferred streams may ask for more than the first one did).
            uint64_t worst9 = 0; for (size_t j : js) worst9 += 9 * chain_bytes(S(j).inflatedLength);
            const bool small = rounds == 0 && i1 == pending.size() && worst <= L.budget / 4;
            { int rc = run_batch(js, small ? worst9 : worst, small ? ~0ull : worst); if (rc) return rc; }
            std::vector<size_t> next;
            for (size_t j : js) if (!prog[j].done) { hard[j] = 1; next.push_back(j); }      // deferred: first in line for the next batch
            if (++rounds > 4 * ns + 16) { ctx->set_err("search batches make no progress"); return ATZ_E_NOMEM; }      // (a stream alone in its batch is never deferred)
            next.insert(next.end(), pending.begin() + i1, pending.end());
            pending.swap(next);
        }
    }
    CK(cudaStreamSynchronize(L.stream));
    return ATZ_OK;
}

// The streams `which` (indices into R) on the search lanes (lane_partition), one host thread each
static int search_set(atz_ctx *ctx, const atz_options *opt, const TrialOpts &topts, std::vector<StreamRec> &R, const std::vector<uint32_t> &which,
                      const std::vector<Params> *seq_class, const std::vector<Params> *seq_brute, const std::vector<Params> *seq_strat) {
    std::vector<uint64_t> ulen(which.size());
    for (size_t k = 0; k < which.size(); k++) ulen[k] = R[which[k]].s.inflatedLength;
    std::vector<std::vector<uint32_t>> part;
    const int nl = lane_partition(ulen.data(), (uint32_t)ulen.size(), getenv("ATZ_LANES") ? atoi(getenv("ATZ_LANES")) : 0, part);
    for (auto &v : part) for (uint32_t &k : v) k = which[k];     // positions in `which` -> indices into R (ascending either way)
    ctx->nlanes_last = nl;
    for (int l = 0; l < nl; l++) { ctx->lane[l].st = atz_stats{}; ctx->lane[l].budget = ctx->budget / nl; }
    std::vector<int> rcs(nl, ATZ_OK);
    {
        std::vector<std::thread> th;
        for (int l = 1; l < nl; l++) th.emplace_back([&, l] { rcs[l] = search_lane(ctx, ctx->lane[l], opt, topts, R, part[l], seq_class, seq_brute, seq_strat); });
        rcs[0] = search_lane(ctx, ctx->lane[0], opt, topts, R, part[0], seq_class, seq_brute, seq_strat);
        for (auto &t : th) t.join();
    }
    for (int l = 0; l < nl; l++) merge_lane_stats(ctx, ctx->lane[l]);   // phase times are per-lane event times and overlap each other
    for (int rc : rcs) if (rc) return rc;
    return ATZ_OK;
}

// One level of the nested descent (ATZ_F_NESTED_DEPTH).  The plaintext P of every parent in `par` (ids as atz_nested.parent counts them)
// is gathered into one scan buffer with ATZ_PAD zero bytes behind each, in batches of at most an eighth of the budget and of 2 GiB (K1's
// candidate positions are 32 bits wide; a batch of one parent, < 0xffffff00 bytes, always fits).  K1 runs over the
// buffer as it is: no accepted first byte is 0x00, and (b0, 0x00) is never a header (b0 * 256 % 31 == 0 only for multiples of 31, none
// of which is accepted), so no hit starts in a gap or runs into one.  K2 inflates every candidate with its input cut at the end of its
// parent (no token map, an output region grown on overflow).  Walking P ascending, a candidate that ends there with a correct adler32
// after more than 16 bytes is a stream, and the walk goes on behind it; no chunking, no IDAT runs.  The streams found are inflated once
// more into regions of their exact size with token maps, as top-level streams are.  Their compressed bytes stay in their parent's P.
static int probe_nested(atz_ctx *ctx, const std::vector<uint64_t> &par, uint32_t depth) {
    const uint64_t ns = ctx->streams.size();
    struct Par { uint64_t id; const uint8_t *plain; uint64_t u; uint32_t owner; };
    std::vector<Par> pv;
    for (uint64_t id : par) { const StreamRec &r = id < ns ? ctx->streams[id] : ctx->nested[id - ns]; pv.push_back(Par{id, r.d_plain, r.s.inflatedLength, r.owner}); }
    const uint32_t flags = ctx->scan_flags & ATZ_SCAN_SMALL_WINDOWS;
    const uint64_t lim = getenv("ATZ_NEST_BATCH") ? (uint64_t)std::max(1, atoi(getenv("ATZ_NEST_BATCH")))     // test hook
                                                  : std::min<uint64_t>(std::max<uint64_t>(ctx->budget / 8, 64ull << 20), 2ull << 30);
    const uint64_t Q = 8192;
    for (size_t b0 = 0; b0 < pv.size();) {
        std::vector<uint64_t> at; uint64_t tot = 0; size_t b1 = b0;
        for (; b1 < pv.size(); b1++) {
            const uint64_t nt = align_up(tot + pv[b1].u + ATZ_PAD, 256);
            if (b1 > b0 && nt > lim) break;
            at.push_back(tot); tot = nt;
        }
        if (at.back() + pv[b1 - 1].u > 0xffffffffull) { ctx->set_err("nested scan buffer positions exceed 32 bits"); return ATZ_E_TOO_LARGE; }
        CK(ctx->nest_scan.ensure(tot + ATZ_PAD));
        uint8_t *buf = ctx->nest_scan.as<uint8_t>();
        CK(cudaMemsetAsync(buf, 0, tot + ATZ_PAD, ctx->stream));
        {
            std::vector<CopyJob> cj;
            for (size_t i = b0; i < b1; i++) if (pv[i].u) cj.push_back(CopyJob{pv[i].plain, buf + at[i - b0], pv[i].u});
            if (!cj.empty()) {
                CK(ctx->cjobs.ensure(cj.size() * sizeof(CopyJob)));
                CK(cudaMemcpyAsync(ctx->cjobs.p, cj.data(), cj.size() * sizeof(CopyJob), cudaMemcpyHostToDevice, ctx->stream));
                CK(launch_gather(ctx->cjobs.as<CopyJob>(), (uint32_t)cj.size(), ctx->stream)); ctx->st.kernel_launches++;
            }
        }
        // ---- K1 over the scan buffer ----
        std::vector<uint32_t> cand; std::vector<uint8_t> ctype;
        {
            Phase ph(ctx, &ctx->st.ms_scan);
            CK(ctx->tile_counts.ensure((size_t)scan_tiles_for(0, tot) * 4 + 64)); CK(ctx->scan_masks.ensure((size_t)scan_tiles_for(0, tot) * 8192 + 64));
            CK(ctx->total.ensure(64)); CK(ctx->queue.ensure(64));
            uint32_t nc = 0;
            CK(launch_scan_count(buf, 0, tot, tot, flags, ctx->tile_counts.as<uint32_t>(), ctx->scan_masks.as<uint16_t>(), ctx->total.as<uint32_t>(), ctx->stream));
            CK(cudaMemcpyAsync(&nc, ctx->total.p, 4, cudaMemcpyDeviceToHost, ctx->stream));
            CK(cudaStreamSynchronize(ctx->stream));
            ctx->st.kernel_launches += 2;
            if (nc) {
                CK(ctx->cand.ensure((size_t)nc * 4)); CK(ctx->ctype.ensure(nc));
                CK(launch_scan_write(buf, 0, tot, ctx->scan_masks.as<uint16_t>(), ctx->tile_counts.as<uint32_t>(), ctx->cand.as<uint32_t>(), ctx->ctype.as<uint8_t>(), nc, ctx->stream));
                ctx->st.kernel_launches++;
                cand.resize(nc); ctype.resize(nc);
                CK(cudaMemcpyAsync(cand.data(), ctx->cand.p, (size_t)nc * 4, cudaMemcpyDeviceToHost, ctx->stream));
                CK(cudaMemcpyAsync(ctype.data(), ctx->ctype.p, nc, cudaMemcpyDeviceToHost, ctx->stream));
            }
            ph.stop();
            CK(cudaGetLastError());
        }
        ctx->st.algo_bytes += tot;
        // ---- K2 probe: every candidate's input is the rest of its parent's P ----
        const size_t nc = cand.size();
        std::vector<uint32_t> pof(nc); std::vector<InflateJob> jobs(nc); std::vector<InflateResult> res(nc);
        for (size_t k = 0, i = 0; k < nc; k++) {
            while (i + 1 < at.size() && cand[k] >= at[i + 1]) i++;
            pof[k] = (uint32_t)i;
            const uint64_t end = at[i] + pv[b0 + i].u, avail = end > cand[k] ? end - cand[k] : 0;
            jobs[k] = InflateJob{cand[k], avail, avail, 0, Q, ~0ull, 0};
        }
        {
            std::vector<size_t> todo(nc); std::vector<uint64_t> cap(nc, Q);
            for (size_t k = 0; k < nc; k++) todo[k] = k;
            while (!todo.empty()) {
                std::vector<size_t> again;
                for (size_t t0 = 0; t0 < todo.size();) {     // launches whose output regions stay within `lim` (at least one job each)
                    std::vector<InflateJob> bj; uint64_t arena = 0; size_t t1 = t0;
                    for (; t1 < todo.size(); t1++) {
                        const uint64_t sz = align_up(cap[todo[t1]] + ATZ_PAD, 256);
                        if (t1 > t0 && arena + sz > lim) break;
                        InflateJob j = jobs[todo[t1]]; j.out_off = arena; j.out_cap = cap[todo[t1]]; bj.push_back(j); arena += sz;
                    }
                    CK(ctx->nest_slots.ensure(arena + ATZ_PAD));
                    CK(cudaMemsetAsync(ctx->nest_slots.p, 0, arena + ATZ_PAD, ctx->stream));
                    std::vector<InflateResult> br, bc;
                    { int rc = run_inflate(ctx, buf, bj, br, bc, ctx->nest_slots.as<uint8_t>(), ~0ull, &ctx->st.ms_inflate_probe); if (rc) return rc; }
                    for (size_t t = t0; t < t1; t++) {
                        const size_t k = todo[t]; res[k] = br[t - t0];
                        // (the bound is deflate's 1032:1 expansion; a plaintext of 4 GiB or more could not be recorded)
                        const uint64_t bound = std::min<uint64_t>(1032 * jobs[k].avail + 65536, 0xffffff00ull);
                        if (res[k].status == INF_OUT_FULL && cap[k] < bound) { cap[k] = std::min<uint64_t>(cap[k] * 6, bound); again.push_back(k); }
                    }
                    t0 = t1;
                }
                todo.swap(again);
            }
        }
        // ---- the walk over each parent's P ----
        std::vector<size_t> acc; uint64_t next = 0;
        for (size_t k = 0, cur = SIZE_MAX; k < nc; k++) {
            if (pof[k] != cur) { cur = pof[k]; next = 0; }
            const uint64_t p = cand[k] - at[pof[k]];
            if (p < next) continue;
            if (res[k].status == INF_END && res[k].total_in > 16 && res[k].total_out < 0xffffff00ull) { acc.push_back(k); next = p + res[k].total_in; }
        }
        // ---- produce mode: plaintext + token map of every stream found ----
        if (!acc.empty()) {
            std::vector<size_t> ord(acc.size());     // longest first (the jobs run off a queue)
            for (size_t i = 0; i < ord.size(); i++) ord[i] = i;
            std::stable_sort(ord.begin(), ord.end(), [&](size_t a, size_t b) { return res[acc[a]].total_out > res[acc[b]].total_out; });
            uint64_t arena = 0; std::vector<InflateJob> vj(acc.size()); std::vector<InflateResult> vr, vc;
            for (size_t i = 0; i < ord.size(); i++) {
                const size_t k = acc[ord[i]]; const uint64_t u = res[k].total_out;
                vj[i] = InflateJob{cand[k], jobs[k].avail, jobs[k].avail, arena, u, 0, 0}; arena = align_up(arena + u + ATZ_PAD, 256);
                vj[i].tmap_off = arena; arena = align_up(arena + u + 64, 256);
            }
            void *q = nullptr; CK(cudaMalloc(&q, arena + ATZ_PAD)); ctx->nest_extra.push_back(q);
            CK(cudaMemsetAsync(q, 0, arena + ATZ_PAD, ctx->stream));
            { int rc = run_inflate(ctx, buf, vj, vr, vc, (uint8_t *)q, ~0ull, &ctx->st.ms_inflate); if (rc) return rc; }
            std::vector<size_t> slot(acc.size());
            for (size_t i = 0; i < ord.size(); i++) slot[ord[i]] = i;
            for (size_t a = 0; a < acc.size(); a++) {
                const size_t k = acc[a], i = slot[a]; const Par &pp = pv[b0 + pof[k]];
                if (vr[i].status != INF_END || vr[i].total_out != res[k].total_out || vr[i].total_in != res[k].total_in) { ctx->set_err("a nested stream inflates differently the second time"); return ATZ_E_DATA; }
                StreamRec r;
                r.s = atz_stream{}; r.s.offset = cand[k] - at[pof[k]]; r.s.streamLength = res[k].total_in; r.s.inflatedLength = res[k].total_out;
                r.s.offsetType = ctype[k]; r.s.clevel = 9; r.s.window = 15; r.s.memlevel = 9; r.s.firstDiffByte = -1;
                r.d_plain = (uint8_t *)q + vj[i].out_off; r.d_tmap = (uint8_t *)q + vj[i].tmap_off; r.d_comp = pp.plain + r.s.offset;
                r.owner = pp.owner; r.adler = vr[i].adler; r.parent = pp.id; r.depth = depth;
                ctx->nested.push_back(std::move(r));
                ctx->st.algo_bytes += res[k].total_in + res[k].total_out;
            }
        }
        b0 = b1;
    }
    return ATZ_OK;
}

int atz_search_shard(atz_ctx *ctx, const atz_options *opt, uint32_t shard, uint32_t nshards) {
    if (!ctx || !opt || nshards == 0 || shard >= nshards) return ATZ_E_ARG;
    const uint32_t depth = (uint32_t)opt->flags >> 8;     // (every bit from 8 up: a depth above 8 is refused, not wrapped)
    if (depth > ATZ_NESTED_MAX) return ATZ_E_ARG;
    if (ctx->state < 2) return ATZ_E_STATE;
    cudaSetDevice(ctx->device);
    drop_nested(ctx);
    const size_t ns = ctx->streams.size();
    const TrialOpts topts = make_opts(opt, true);
    ctx->dbg = HostDbg{}; for (int l = 0; l < ATZ_LANES; l++) ctx->lane[l].dbg = &ctx->dbg;
    ctx->dbg.lanes = getenv("ATZ_DEBUG_LANES") != nullptr; ctx->dbg.t0 = ctx->dbg.t = std::chrono::steady_clock::now(); host_mark(ctx->lane[0], -1);
    // the candidate sequences depend on the header type only: built once per type, shared by the streams
    static std::vector<Params> seq_class[ATZ_NTYPES], seq_brute[ATZ_NTYPES], seq_strat[ATZ_NTYPES];
    static std::once_flag seq_once;
    std::call_once(seq_once, [] { for (int ty = 0; ty < ATZ_NTYPES; ty++) { class_sequence(ty, seq_class[ty]); brute_sequence(ty, seq_brute[ty]); strategy_sequence(ty, seq_strat[ty]); } });
    // which streams this call searches: after a sharded scan the ones this context owns (it holds no other plaintext); after a
    // plain atz_scan any partition can be asked for (every stream is resident) and is computed the same way (atz_host_partition)
    if (ctx->sc.nshards > 1 && (nshards != ctx->sc.nshards || shard != ctx->sc.shard)) { ctx->set_err("atz_search_shard: shard does not match the sharded scan"); return ATZ_E_ARG; }
    if (ctx->sc.nshards == 1) {
        std::vector<uint64_t> ul(ns); std::vector<uint32_t> ow(ns, 0);
        for (size_t s = 0; s < ns; s++) ul[s] = ctx->streams[s].s.inflatedLength;
        stream_partition(ul.data(), nullptr, (uint32_t)ns, nshards, ow.data());
        for (size_t s = 0; s < ns; s++) ctx->streams[s].owner = ow[s];
    }
    std::vector<uint32_t> mine;
    for (size_t s = 0; s < ns; s++) {
        StreamRec &r = ctx->streams[s];
        r.s.identBytes = 0; r.s.clevel = 9; r.s.window = 15; r.s.memlevel = 9; r.s.recomp = 0; r.s.firstDiffByte = -1; r.s.ndiff = 0; r.diff_off.clear(); r.diff_val.clear();
        if (r.owner == shard) mine.push_back((uint32_t)s);
    }
    { int rc = search_set(ctx, opt, topts, ctx->streams, mine, seq_class, seq_brute, seq_strat); if (rc) return rc; }
    // ATZ_F_NESTED_DEPTH: level by level, the plaintext of the recompressed streams of the level above that this context owns is scanned
    // (probe_nested) and the streams found there are searched like top-level ones; they belong to their parent's owner
    std::vector<uint64_t> par;
    for (size_t s = 0; s < ns && depth; s++) if (ctx->streams[s].s.recomp && ctx->streams[s].owner == shard && ctx->streams[s].d_plain) par.push_back(s);
    for (uint32_t d = 1; d <= depth && !par.empty(); d++) {
        const size_t first = ctx->nested.size();
        {   // the scan buffer and the probe slots are needed for the probe only
            const int rc = probe_nested(ctx, par, d);
            ctx->nest_scan.release(); ctx->nest_slots.release();
            if (rc) return rc;
        }
        std::vector<uint32_t> lvl;
        for (size_t j = first; j < ctx->nested.size(); j++) lvl.push_back((uint32_t)j);
        { int rc = search_set(ctx, opt, topts, ctx->nested, lvl, seq_class, seq_brute, seq_strat); if (rc) return rc; }
        par.clear();
        for (uint32_t j : lvl) if (ctx->nested[j].s.recomp) par.push_back(ns + j);
    }
    uint64_t di = 0, nrec = 0, atz = 28, lastend = 0;
    for (auto &r : ctx->streams) {
        r.s.diff_index = di; di += r.s.ndiff;
        if (r.s.recomp) { nrec++; atz += 35 + (r.s.ndiff ? 8 + 9 * r.s.ndiff : 0) + r.s.inflatedLength + (r.pieces.empty() ? 0 : 8 + 4 * r.pieces.size() + (uint64_t)r.frame * (r.pieces.size() - 1)); }
        else atz += r.span();
        if (r.s.offset >= lastend) { atz += r.s.offset - lastend; }
        lastend = r.s.offset + r.span();
    }
    if (lastend < ctx->n) atz += ctx->n - lastend;
    for (auto &r : ctx->nested) { r.s.diff_index = di; di += r.s.ndiff; }
    ctx->st.n_recomp = nrec;
    ctx->st.algo_bytes += ctx->st.trial_algo_bytes + atz;
    host_mark(ctx->lane[0], 0);
    if (getenv("ATZ_DEBUG_HOST")) fprintf(stderr, "[host ms, lane 0] requests+fold %.1f | chains prep %.1f | rows prep %.1f | resolve prep %.1f | sort+descs %.1f | launch+results %.1f\n", ctx->dbg.ms[0], ctx->dbg.ms[1], ctx->dbg.ms[2], ctx->dbg.ms[3], ctx->dbg.ms[4], ctx->dbg.ms[5]);
    ctx->state = 3;
    return ATZ_OK;
}

int atz_get_streams(atz_ctx *ctx, atz_stream *streams, uint64_t cap) {
    if (!ctx || (!streams && cap)) return ATZ_E_ARG;
    if (ctx->state < 2) return ATZ_E_STATE;
    if (cap < ctx->streams.size()) return ATZ_E_SMALL;
    for (size_t i = 0; i < ctx->streams.size(); i++) streams[i] = ctx->streams[i].s;
    return ATZ_OK;
}
int atz_get_owners(atz_ctx *ctx, uint32_t *owner, uint64_t cap) {
    if (!ctx || (!owner && cap)) return ATZ_E_ARG;
    if (ctx->state < 2) return ATZ_E_STATE;
    if (cap < ctx->streams.size()) return ATZ_E_SMALL;
    for (size_t i = 0; i < ctx->streams.size(); i++) owner[i] = ctx->streams[i].owner;
    return ATZ_OK;
}
int atz_get_pieces(atz_ctx *ctx, uint64_t i, uint32_t *len, uint64_t cap, uint64_t *npieces) {
    if (!ctx || !npieces || (!len && cap)) return ATZ_E_ARG;
    if (ctx->state < 2) return ATZ_E_STATE;
    if (i >= ctx->streams.size()) return ATZ_E_ARG;
    const std::vector<uint32_t> &p = ctx->streams[i].pieces;
    *npieces = p.size();
    if (cap < p.size()) return ATZ_E_SMALL;
    if (!p.empty()) memcpy(len, p.data(), p.size() * 4);
    return ATZ_OK;
}
int atz_get_framing(atz_ctx *ctx, uint64_t i, uint32_t *bytes) {
    if (!ctx || !bytes) return ATZ_E_ARG;
    if (ctx->state < 2) return ATZ_E_STATE;
    if (i >= ctx->streams.size()) return ATZ_E_ARG;
    *bytes = ctx->streams[i].pieces.empty() ? 0 : ctx->streams[i].frame;
    return ATZ_OK;
}
int atz_get_diffs(atz_ctx *ctx, uint64_t *offsets, uint8_t *values, uint64_t cap, uint64_t *n) {
    if (!ctx) return ATZ_E_ARG;
    if (ctx->state < 3) return ATZ_E_STATE;
    uint64_t tot = 0; for (auto &r : ctx->streams) tot += r.s.ndiff;
    for (auto &r : ctx->nested) tot += r.s.ndiff;
    if (n) *n = tot;
    if (cap < tot) return ATZ_E_SMALL;
    uint64_t o = 0;
    for (auto *v : {&ctx->streams, &ctx->nested})
        for (auto &r : *v) for (uint64_t i = 0; i < r.s.ndiff; i++) { offsets[o] = r.diff_off[i]; values[o] = r.diff_val[i]; o++; }
    return ATZ_OK;
}
int atz_get_nested(atz_ctx *ctx, atz_nested *out, uint64_t cap, uint64_t *n) {
    if (!ctx || !n || (!out && cap)) return ATZ_E_ARG;
    if (ctx->state < 3) return ATZ_E_STATE;
    *n = ctx->nested.size();
    if (cap < ctx->nested.size()) return ATZ_E_SMALL;
    for (size_t j = 0; j < ctx->nested.size(); j++) { const StreamRec &r = ctx->nested[j]; out[j] = atz_nested{r.parent, r.depth, 0, r.s}; }
    return ATZ_OK;
}
// stream i as atz_get_inflated counts: top-level streams, then the nested ones (nullptr: no such stream)
static StreamRec *stream_at(atz_ctx *ctx, uint64_t i) {
    const uint64_t ns = ctx->streams.size();
    return i < ns ? &ctx->streams[i] : i - ns < ctx->nested.size() ? &ctx->nested[i - ns] : nullptr;
}
int atz_get_inflated(atz_ctx *ctx, uint64_t i, uint8_t *dst, uint64_t cap) {
    if (!ctx || !dst) return ATZ_E_ARG;
    if (ctx->state < 2) return ATZ_E_STATE;
    StreamRec *rp = stream_at(ctx, i);
    if (!rp) return ATZ_E_ARG;
    StreamRec &r = *rp;
    if (cap < r.s.inflatedLength) return ATZ_E_SMALL;
    if (!r.d_plain) { ctx->set_err("stream is owned by another shard"); return ATZ_E_STATE; }
    cudaSetDevice(ctx->device);
    Phase ph(ctx, &ctx->st.ms_d2h);
    CK(cudaMemcpyAsync(dst, r.d_plain, r.s.inflatedLength, cudaMemcpyDeviceToHost, ctx->stream));
    ph.stop();
    return ATZ_OK;
}
static int gather_streams(atz_ctx *ctx, const std::vector<const StreamRec *> &which, uint8_t *dst, uint64_t tot) {
    // the payloads go into one contiguous device buffer (one kernel), then a single D2H copy
    CK(ctx->gather.ensure(tot + 64)); CK(ctx->cjobs.ensure(which.size() * sizeof(CopyJob)));
    std::vector<CopyJob> cj; cj.reserve(which.size());
    uint64_t o = 0;
    for (const StreamRec *p : which) { const StreamRec &r = *p; cj.push_back(CopyJob{r.d_plain, ctx->gather.as<uint8_t>() + o, r.s.inflatedLength}); o += r.s.inflatedLength; }
    CK(cudaMemcpyAsync(ctx->cjobs.p, cj.data(), cj.size() * sizeof(CopyJob), cudaMemcpyHostToDevice, ctx->stream));
    Phase ph(ctx, &ctx->st.ms_d2h);
    CK(launch_gather(ctx->cjobs.as<CopyJob>(), (uint32_t)cj.size(), ctx->stream)); ctx->st.kernel_launches++;
    CK(cudaMemcpyAsync(dst, ctx->gather.p, tot, cudaMemcpyDeviceToHost, ctx->stream));
    ph.stop();
    return ATZ_OK;
}
int atz_get_inflated_recomp(atz_ctx *ctx, uint8_t *dst, uint64_t cap, uint64_t *n) {
    if (!ctx) return ATZ_E_ARG;
    if (ctx->state < 3) return ATZ_E_STATE;
    uint64_t tot = 0; std::vector<const StreamRec *> which;
    for (const StreamRec &r : ctx->streams) if (r.s.recomp && r.d_plain) { tot += r.s.inflatedLength; which.push_back(&r); }   // (of a sharded run: the ones this context owns)
    if (n) *n = tot;
    if (!dst || cap < tot) return ATZ_E_SMALL;
    if (!tot) return ATZ_OK;
    cudaSetDevice(ctx->device);
    return gather_streams(ctx, which, dst, tot);
}
int atz_get_inflated_list(atz_ctx *ctx, const uint64_t *indices, uint64_t count, uint8_t *dst, uint64_t cap, uint64_t *n) {
    if (!ctx || (!indices && count)) return ATZ_E_ARG;
    if (ctx->state < 2) return ATZ_E_STATE;
    uint64_t tot = 0; std::vector<const StreamRec *> which;
    for (uint64_t k = 0; k < count; k++) {
        const StreamRec *r = stream_at(ctx, indices[k]);
        if (!r) return ATZ_E_ARG;
        if (!r->d_plain) { ctx->set_err("stream is owned by another shard"); return ATZ_E_STATE; }
        tot += r->s.inflatedLength; which.push_back(r);
    }
    if (n) *n = tot;
    if (!dst || cap < tot) return ATZ_E_SMALL;
    if (!tot) return ATZ_OK;
    cudaSetDevice(ctx->device);
    return gather_streams(ctx, which, dst, tot);
}
int atz_timer_start(atz_ctx *ctx) {
    if (!ctx) return ATZ_E_ARG;
    cudaSetDevice(ctx->device);
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaEventRecord(ctx->tev0, ctx->stream));
    return ATZ_OK;
}
int atz_timer_stop(atz_ctx *ctx, double *ms) {
    if (!ctx || !ms) return ATZ_E_ARG;
    cudaSetDevice(ctx->device);
    CK(cudaEventRecord(ctx->tev1, ctx->stream));
    CK(cudaEventSynchronize(ctx->tev1));
    float f = 0; CK(cudaEventElapsedTime(&f, ctx->tev0, ctx->tev1)); *ms = f;
    return ATZ_OK;
}
int atz_get_stats(atz_ctx *ctx, atz_stats *st) { if (!ctx || !st) return ATZ_E_ARG; *st = ctx->st; return ATZ_OK; }

// ---------------------------------------------------------------------------------------------
// single-stream operators
static int upload_padded(atz_ctx *ctx, Buf &b, const uint8_t *src, uint64_t n, uint64_t lead = 0) {
    CK(b.ensure(lead + n + 2 * ATZ_PAD));
    CK(cudaMemsetAsync(b.p, 0, lead + n + 2 * ATZ_PAD, ctx->stream));
    if (n) CK(cudaMemcpyAsync(b.as<uint8_t>() + lead, src, n, cudaMemcpyHostToDevice, ctx->stream));
    return ATZ_OK;
}
static int device_adler(atz_ctx *ctx, const std::vector<AdlerJob> &jobs) {
    Lane &L = ctx->lane[0];
    CK(L.djobs.ensure(jobs.size() * sizeof(AdlerJob)));
    CK(cudaMemcpyAsync(L.djobs.p, jobs.data(), jobs.size() * sizeof(AdlerJob), cudaMemcpyHostToDevice, ctx->stream));
    CK(launch_adler(L.djobs.as<AdlerJob>(), (uint32_t)jobs.size(), ctx->stream));
    ctx->st.kernel_launches++;
    return ATZ_OK;
}

int atz_deflate_batch(atz_ctx *ctx, const uint8_t *in, const uint64_t *in_off, const uint64_t *in_len, const uint8_t *clevel, const uint8_t *window,
                      const uint8_t *memlevel, uint64_t n, uint8_t *out, const uint64_t *out_off, const uint64_t *out_cap, uint64_t *out_len) {
    if (!ctx || !in_off || !in_len || !clevel || !window || !memlevel || !out || !out_off || !out_cap || !out_len) return ATZ_E_ARG;
    if (n == 0) return ATZ_OK;
    cudaSetDevice(ctx->device);
    uint64_t tot_in = 0, tot_out = 0, worst = 0, lo = ~0ull, hi = 0, sum_in = 0;
    std::vector<uint64_t> din(n), dout(n);
    for (uint64_t i = 0; i < n; i++) {
        if ((clevel[i] & 15) > 9 || (clevel[i] >> 4) > 4 || window[i] < 9 || window[i] > 15 || memlevel[i] < 1 || memlevel[i] > 9) return ATZ_E_ARG;
        if (in_len[i] >= 0xffffff00ull) return ATZ_E_TOO_LARGE;
        din[i] = tot_in; tot_in = align_up(tot_in + in_len[i] + ATZ_PAD, 256);
        dout[i] = tot_out; tot_out = align_up(tot_out + out_cap[i] + 8, 256);
        if (needs_chain(Params{(uint8_t)(clevel[i] & 15), window[i], memlevel[i], (uint8_t)(clevel[i] >> 4)})) worst += chain_bytes(in_len[i]);
        if (in_len[i]) { lo = std::min(lo, in_off[i]); hi = std::max(hi, in_off[i] + in_len[i]); sum_in += in_len[i]; }
    }
    // inputs that sit close together in the caller's buffer (the payloads of an ATZ file, main.cpp:893-913) are uploaded as one span
    // and read in place - the kernels accept any alignment and only need readable slack behind each input; otherwise one copy each
    const bool one_span = sum_in && (hi - lo) <= sum_in + sum_in / 4 + (1u << 20);
    if (one_span) { tot_in = align_up(hi - lo + ATZ_PAD, 256); for (uint64_t i = 0; i < n; i++) din[i] = in_len[i] ? in_off[i] - lo : 0; }
    CK(ctx->op_in.ensure(tot_in + ATZ_PAD)); CK(ctx->op_out.ensure(tot_out + 256)); CK(ctx->op_misc.ensure(n * 4 + 64));
    {
        Phase ph(ctx, &ctx->st.ms_h2d);
        if (one_span) {
            CK(cudaMemcpyAsync(ctx->op_in.p, in + lo, hi - lo, cudaMemcpyHostToDevice, ctx->stream));
            CK(cudaMemsetAsync(ctx->op_in.as<uint8_t>() + (hi - lo), 0, tot_in + ATZ_PAD - (hi - lo), ctx->stream));
        } else {
            CK(cudaMemsetAsync(ctx->op_in.p, 0, tot_in + ATZ_PAD, ctx->stream));
            for (uint64_t i = 0; i < n; i++) if (in_len[i]) CK(cudaMemcpyAsync(ctx->op_in.as<uint8_t>() + din[i], in + in_off[i], in_len[i], cudaMemcpyHostToDevice, ctx->stream));
        }
        ph.stop();
    }
    std::vector<AdlerJob> aj(n);
    for (uint64_t i = 0; i < n; i++) aj[i] = AdlerJob{ctx->op_in.as<uint8_t>() + din[i], (uint32_t)in_len[i], ctx->op_misc.as<uint32_t>() + i};
    { int rc = device_adler(ctx, aj); if (rc) return rc; }
    std::vector<uint32_t> ad(n);
    CK(cudaMemcpyAsync(ad.data(), ctx->op_misc.p, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    Lane &L = ctx->lane[0]; L.budget = ctx->budget; L.st = atz_stats{};
    { int rc = chain_arena_for(ctx, L, worst); if (rc) return rc; }
    { uint64_t rw = 0; for (uint64_t i = 0; i < n; i++) if ((clevel[i] & 15) >= 4) rw += 40 * (in_len[i] + 64) + 1024; if (rw) rec_arena_for(ctx, L, rw); }
    // process in groups that fit the chain arena
    uint64_t i0 = 0;
    while (i0 < n) {
        uint64_t i1 = i0, used = 0;
        while (i1 < n) { uint64_t a = chain_bytes(in_len[i1]); if (i1 > i0 && used + a > L.chains.cap) break; used += a; i1++; }   // (an upper bound: strategies 2 and 3 need none)
        std::vector<PlainView> views; std::vector<TrialReq> reqs;
        for (uint64_t i = i0; i < i1; i++) {
            views.push_back(PlainView{ctx->op_in.as<uint8_t>() + din[i], (uint32_t)in_len[i], nullptr, 0, ad[i]});
            uint32_t cap4 = (uint32_t)std::min<uint64_t>(align_up(out_cap[i], 4), 0xfffffff0u);
            { TrialReq rq{(uint32_t)(i - i0), Params{(uint8_t)(clevel[i] & 15), window[i], memlevel[i], (uint8_t)(clevel[i] >> 4)}, 1, ctx->op_out.as<uint8_t>() + dout[i], cap4};
              if (rq.prm.c >= 4 && needs_chain(rq.prm)) { rq.want_rec = 2; rq.want_res = 1; }
              reqs.push_back(rq); }
        }
        ChainState cs; std::vector<TrialResult> tr;
        TrialOpts so = make_opts(nullptr, false);
        { int rc = run_trials(ctx, L, views, reqs, so, cs, tr); merge_lane_stats(ctx, L); if (rc) return rc; }
        Phase ph(ctx, &ctx->st.ms_d2h);
        for (uint64_t i = i0; i < i1; i++) {
            const TrialResult &r = tr[i - i0];
            out_len[i] = r.out_len;
            if (r.status == TR_OVERFLOW || r.out_len > out_cap[i]) return ATZ_E_SMALL;
            CK(cudaMemcpyAsync(out + out_off[i], ctx->op_out.as<uint8_t>() + dout[i], r.out_len, cudaMemcpyDeviceToHost, ctx->stream));
        }
        ph.stop();
        i0 = i1;
    }
    CK(cudaStreamSynchronize(ctx->stream));
    return ATZ_OK;
}

int atz_deflate_stream(atz_ctx *ctx, const uint8_t *in, uint64_t n, int clevel, int window, int memlevel, uint8_t *out, uint64_t cap, uint64_t *out_len) {
    if (!ctx || (!in && n) || !out || !out_len) return ATZ_E_ARG;
    if (clevel < 0 || (clevel & 15) > 9 || (clevel >> 4) > 4 || window < 9 || window > 15 || memlevel < 1 || memlevel > 9) return ATZ_E_ARG;
    uint64_t io = 0, oo = 0; uint8_t c = (uint8_t)clevel, w = (uint8_t)window, m = (uint8_t)memlevel;
    static const uint8_t dummy = 0;
    return atz_deflate_batch(ctx, in ? in : &dummy, &io, &n, &c, &w, &m, 1, out, &oo, &cap, out_len);
}

int atz_inflate_stream(atz_ctx *ctx, const uint8_t *in, uint64_t n, uint8_t *out, uint64_t cap, uint64_t *out_len, uint64_t *consumed) {
    if (!ctx || !in || (!out && cap)) return ATZ_E_ARG;
    if (n >= 0xffffff00ull) return ATZ_E_TOO_LARGE;
    cudaSetDevice(ctx->device);
    { int rc = upload_padded(ctx, ctx->op_orig, in, n); if (rc) return rc; }
    // zlib fills the caller's buffer to the last byte (a match is cut where the room ends) and reports the input it has consumed by
    // then; the kernel produces whole tokens, so it gets some slack behind `cap` and tells how much input was used when the output
    // first reached `cap` (the scan kernel's in_at_outcap, checked against zlib in tests/test_gpu_kernels.py)
    const uint64_t cap2 = cap + 65536 + 512;     // (a stored block of up to 65535 bytes is copied whole or not at all)
    CK(ctx->op_out.ensure(cap2 + ATZ_PAD)); CK(ctx->jobs.ensure(sizeof(InflateJob))); CK(ctx->jres.ensure(sizeof(InflateResult))); CK(ctx->jres2.ensure(sizeof(InflateResult))); CK(ctx->queue.ensure(64));
    InflateJob j{0, n, n, 0, cap2, ~0ull}; InflateResult r{};
    CK(cudaMemcpyAsync(ctx->jobs.p, &j, sizeof j, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemsetAsync(ctx->queue.p, 0, 4, ctx->stream));
    {
        Phase ph(ctx, &ctx->st.ms_inflate);
        CK(launch_inflate(ctx->op_orig.as<uint8_t>(), ctx->jobs.as<InflateJob>(), ctx->jres.as<InflateResult>(), ctx->jres2.as<InflateResult>(), 1, ctx->queue.as<uint32_t>(),
                          ctx->op_out.as<uint8_t>(), cap, 2, 1, 1, ctx->stream));
        ph.stop(); ctx->st.kernel_launches++;
    }
    CK(cudaMemcpyAsync(&r, ctx->jres.p, sizeof r, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    const bool full = r.total_out > cap;     // more output than the caller has room for: what zlib reports at that point
    if (out_len) *out_len = full ? cap : r.total_out;
    if (consumed) *consumed = full ? r.in_at_outcap : r.total_in;
    uint64_t give = std::min<uint64_t>(r.total_out, cap);
    if (give) CK(cudaMemcpy(out, ctx->op_out.p, give, cudaMemcpyDeviceToHost));
    if (full || r.status == INF_OUT_FULL) return ATZ_E_SMALL;
    if (r.status == INF_NEED_INPUT) return ATZ_E_TRUNCATED;
    if (r.status != INF_END) return ATZ_E_DATA;
    return ATZ_OK;
}

int atz_trial(atz_ctx *ctx, const uint8_t *in, uint64_t n, const uint8_t *orig, uint64_t c, int clevel, int window, int memlevel,
              const atz_options *opt, atz_trial_result *res) {
    if (!ctx || (!in && n) || !orig || !opt || !res) return ATZ_E_ARG;
    if (clevel < 0 || (clevel & 15) > 9 || (clevel >> 4) > 4 || window < 9 || window > 15 || memlevel < 1 || memlevel > 9) return ATZ_E_ARG;
    if (n >= 0xffffff00ull || c >= 0xffffff00ull) return ATZ_E_TOO_LARGE;
    cudaSetDevice(ctx->device);
    { int rc = upload_padded(ctx, ctx->op_in, in, n); if (rc) return rc; }
    { int rc = upload_padded(ctx, ctx->op_orig, orig, c, 16); if (rc) return rc; }
    CK(ctx->op_misc.ensure(64)); CK(ctx->queue.ensure(64));
    std::vector<AdlerJob> aj{AdlerJob{ctx->op_in.as<uint8_t>(), (uint32_t)n, ctx->op_misc.as<uint32_t>()}};
    { int rc = device_adler(ctx, aj); if (rc) return rc; }
    uint32_t ad = 0;
    CK(cudaMemcpyAsync(&ad, ctx->op_misc.p, 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    Lane &L = ctx->lane[0]; L.budget = ctx->budget; L.st = atz_stats{};
    { int rc = chain_arena_for(ctx, L, chain_bytes(n)); if (rc) return rc; }
    rec_arena_for(ctx, L, 40 * (n + 64) + 4096);
    std::vector<PlainView> views{PlainView{ctx->op_in.as<uint8_t>(), (uint32_t)n, ctx->op_orig.as<uint8_t>() + 16, (uint32_t)c, ad}};
    std::vector<TrialReq> reqs{TrialReq{0, Params{(uint8_t)(clevel & 15), (uint8_t)window, (uint8_t)memlevel, (uint8_t)(clevel >> 4)}, 0, nullptr, 0}};
    if (needs_chain(reqs[0].prm)) { reqs[0].want_rec = 2; reqs[0].want_res = 1; }
    ChainState cs; std::vector<TrialResult> tr;
    { int rc = run_trials(ctx, L, views, reqs, make_opts(opt, true), cs, tr); merge_lane_stats(ctx, L); if (rc) return rc; }
    res->status = tr[0].status; res->in_consumed = tr[0].in_consumed; res->out_len = tr[0].out_len; res->ident = tr[0].ident;
    res->kcycles = tr[0].kcycles; res->kcycles_flush = tr[0].kcycles_flush;
    return ATZ_OK;
}

// ---- host-logic test hooks: pure host code, usable without a CUDA device (tests/test_host_logic.py) ----
int atz_host_header_type(uint32_t scan_flags, uint32_t b0, uint32_t b1) { return zlib_header_type(b0 & 0xff, b1 & 0xff, scan_flags); }
int atz_host_idat_run(const uint8_t *file, uint64_t n, uint64_t p, uint32_t *len, uint64_t cap, uint64_t *npieces) {
    if (!file || !npieces || (!len && cap)) return ATZ_E_ARG;
    *npieces = p < n ? idat_run(file, n, 0, n, p, len, (uint32_t)std::min<uint64_t>(cap, 0xffffffffull)) : 0;
    return ATZ_OK;
}
int atz_host_fdat_run(const uint8_t *file, uint64_t n, uint64_t p, uint32_t *len, uint64_t cap, uint64_t *npieces) {
    if (!file || !npieces || (!len && cap)) return ATZ_E_ARG;
    *npieces = p < n ? fdat_run(file, n, 0, n, p, len, (uint32_t)std::min<uint64_t>(cap, 0xffffffffull)) : 0;
    return ATZ_OK;
}
int atz_host_candidate_sequence(int offsetType, int brute, uint8_t *clevel, uint8_t *window, uint8_t *memlevel, uint32_t cap) {
    if (offsetType < 0 || offsetType >= ATZ_NTYPES) return ATZ_E_ARG;
    std::vector<Params> v;
    if (brute == 2) strategy_sequence(offsetType, v); else if (brute) brute_sequence(offsetType, v); else class_sequence(offsetType, v);
    for (size_t i = 0; i < v.size() && i < cap; i++) { clevel[i] = (uint8_t)(v[i].c | (v[i].s << 4)); window[i] = v[i].w; memlevel[i] = v[i].m; }
    return (int)v.size();
}
/* lane_of[k] receives the search lane of the k-th stream of a shard, given the streams' inflated lengths; returns the number of lanes */
int atz_host_lane_partition(const uint64_t *inflated_len, uint32_t n, int forced_lanes, uint32_t *lane_of) {
    if ((!inflated_len || !lane_of) && n) return ATZ_E_ARG;
    std::vector<std::vector<uint32_t>> part;
    const int nl = lane_partition(inflated_len, n, forced_lanes, part);
    for (int l = 0; l < nl; l++) for (uint32_t k : part[l]) lane_of[k] = (uint32_t)l;
    return nl;
}
int atz_host_partition(const uint64_t *inflated_len, const uint32_t *probed_by, uint32_t n, uint32_t nshards, uint32_t *owner) {
    if ((!inflated_len || !owner) && n) return ATZ_E_ARG;
    if (nshards == 0) return ATZ_E_ARG;
    stream_partition(inflated_len, probed_by, n, nshards, owner);
    return ATZ_OK;
}
int atz_host_chunks(uint64_t n, uint64_t chunksize, uint64_t *start, uint64_t *len, uint64_t cap) {
    if (n == 0 || chunksize < 2) return ATZ_E_ARG;
    std::vector<uint64_t> cs, cl; chunk_list(n, chunksize, cs, cl);
    for (size_t i = 0; i < cs.size() && i < cap; i++) { start[i] = cs[i]; len[i] = cl[i]; }
    return (int)cs.size();
}
/* records: {status, total_in, total_out, in_at_outcap} as 4 x uint64 per candidate (status: 0 END, 1 NEED_INPUT, 2 DATA_ERROR).
 * out: up to cap accepted streams as {offset, total_in, total_out}.  Returns the number accepted. */
int atz_host_scan_fold(uint64_t n, uint64_t chunksize, const uint32_t *cand, uint32_t ncand, const uint64_t *probe, const uint64_t *avail,
                       const int32_t *cont_of, const uint64_t *cont, uint32_t ncont, uint64_t *out, uint32_t cap) {
    if (n == 0 || chunksize < 2) return ATZ_E_ARG;
    std::vector<uint64_t> cs, cl; chunk_list(n, chunksize, cs, cl);
    std::vector<ProbeRec> pr(ncand), cr(ncont);
    for (uint32_t k = 0; k < ncand; k++) pr[k] = ProbeRec{(int32_t)probe[4 * k], probe[4 * k + 1], probe[4 * k + 2], probe[4 * k + 3]};
    for (uint32_t k = 0; k < ncont; k++) cr[k] = ProbeRec{(int32_t)cont[4 * k], cont[4 * k + 1], cont[4 * k + 2], cont[4 * k + 3]};
    std::vector<Acc> acc;
    scan_fold(cs, cl, cand, ncand, pr.data(), avail, cont_of, cr.data(), acc);
    for (size_t i = 0; i < acc.size() && i < cap; i++) { out[3 * i] = acc[i].off; out[3 * i + 1] = acc[i].tin; out[3 * i + 2] = acc[i].tout; }
    return (int)acc.size();
}

} // extern "C"

// uncomp - the AntiZ command line on top of the antiz_b200 C ABI.
//
// Drop-in for the reference's `uncomp` (reference: /root/reference/main.cpp): same flags and defaults
// (parseCLI main.cpp:1070-1143), same stdout lines (main.cpp:268,291,295,798,875-879,1178,1196), same ATZ1 bytes
// (writeATZfile/writeStreamdesc main.cpp:764-831), same reconstruction (reconstructATZ main.cpp:869-950) and the
// same built-in self test (testATZfile main.cpp:1173-1203).  The host keeps what the reference's L1/L2 layers do
// (CLI, file IO, ATZ1 layout, phase order); phases 1 and 3 and the per-stream deflate of the reconstructor run on
// the GPU.  Extensions: --gpus N (static shard of the stream x parameter grid), --device D, --exact-records, --stats, --strategies,
// --small-windows, --png, --nested, --apng.
#include "ATZData.h"
#include "antiz_b200.h"
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <iostream>
#include <string>
#include <thread>
#include <algorithm>
#include <vector>
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#define antiz_ver "0.1.6-git"

namespace {

bool read_file(const std::string &name, std::vector<uint8_t> &buf) {
    std::ifstream f(name, std::ios::in | std::ios::binary);
    if (!f.is_open()) return false;
    f.seekg(0, f.end); std::streamoff n = f.tellg(); f.seekg(0, f.beg);
    buf.resize((size_t)n);
    if (n) f.read(reinterpret_cast<char *>(buf.data()), n);
    return true;
}
int getFilesize(const std::string &fname, uint64_t &fsize) {   // main.cpp:27-41
    std::ifstream f(fname, std::ios::in | std::ios::binary);
    if (!f.is_open()) {
        std::cout << "error: open file for size check failed!" << std::endl;
        std::cout << "Cannot open file: " << fname << std::endl;
        return -1;
    }
    f.seekg(0, f.end); fsize = (uint64_t)f.tellg();
    return 0;
}
inline void put8(std::vector<uint8_t> &o, uint64_t v) { for (int i = 0; i < 8; i++) o.push_back((uint8_t)(v >> (8 * i))); }   // writeNumber8: raw little-endian u64
inline uint64_t get8(const uint8_t *p) { uint64_t v; std::memcpy(&v, p, 8); return v; }
const char *atz_err(atz_ctx *c, int rc) { static std::string s; s = "antiz_b200 error " + std::to_string(rc) + ": " + (c ? atz_last_error(c) : ""); return s.c_str(); }

// The input file, mapped read-only: nothing is copied into a buffer of the program's own (the reference reads it chunk by chunk,
// main.cpp:392-420, and again per stream, main.cpp:431-436); the library uploads from the mapping what each GPU needs.
struct MappedFile {
    const uint8_t *p = nullptr; size_t n = 0; int fd = -1;
    bool open(const std::string &name) {
        fd = ::open(name.c_str(), O_RDONLY);
        if (fd < 0) return false;
        struct stat st;
        if (fstat(fd, &st) != 0) return false;
        n = (size_t)st.st_size;
        if (n) {
            void *m = mmap(nullptr, n, PROT_READ, MAP_PRIVATE | MAP_POPULATE, fd, 0);
            if (m == MAP_FAILED) return false;
            p = (const uint8_t *)m;
            madvise(m, n, MADV_SEQUENTIAL);
        }
        return true;
    }
    const uint8_t *data() const { return p; }
    size_t size() const { return n; }
    const uint8_t *begin() const { return p; }
    const uint8_t *end() const { return p + n; }
    ~MappedFile() { if (p) munmap((void *)p, n); if (fd >= 0) ::close(fd); }
};

struct Timer { std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now(); double ms() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count(); } };

} // namespace

// ---------------------------------------------------------------------------------------------
// ATZcreator: same phase protocol as the reference (main.cpp:252-308); -10 on a phase out of order.
class ATZcreator {
  public:
    ATZcreator(const std::string ifname, const std::string atzname, const std::string recname, const ATZdata::programOptions opt)
        : infileName(ifname), atzfileName(atzname), reconfileName(recname), options(opt) {}
    ~ATZcreator() { for (auto c : ctxs) atz_ctx_destroy(c); }

    int Phase1() {   // scan + trial inflate (searchInfile + ZBuffSearcher)
        if (processingState != 0) return -10;
        if (!file.open(infileName)) { std::cerr << "Error Encountered: failed to open File " << infileName << std::endl; std::exit(1); }
        infileSize = file.size();
        int ng = options.gpus < 1 ? 1 : options.gpus;
        ctxs.assign(ng, nullptr);
        {   // the contexts are created side by side: a primary context per device is seconds of driver work on an 8-GPU box
            static const bool one_device = getenv("ATZ_TEST_ONE_DEVICE") != nullptr;   // test hook: every shard on the first device
            std::vector<int> crc(ng, ATZ_OK);
            auto mk = [&](int g) { crc[g] = atz_ctx_create(one_device ? options.device : options.device + g, &ctxs[g]); };
            std::vector<std::thread> th;
            for (int g = 1; g < ng; g++) th.emplace_back(mk, g);
            mk(0);
            for (auto &t : th) t.join();
            for (int g = 0; g < ng; g++) if (crc[g] != ATZ_OK) { std::cout << "error: no usable CUDA device " << (options.device + g) << " (antiz_b200 has no CPU path)" << std::endl; std::exit(1); }
            const uint32_t scan_flags = (options.smallWindows ? ATZ_SCAN_SMALL_WINDOWS : 0) | (options.png ? ATZ_SCAN_PNG_IDAT : 0) | (options.apng ? ATZ_SCAN_APNG_FDAT : 0);
            for (int g = 0; g < ng && scan_flags; g++) {   // before any load: every shard scans with the same header set
                const int rc = atz_ctx_set_scan_flags(ctxs[g], scan_flags);
                if (rc != ATZ_OK) { std::cout << atz_err(ctxs[g], rc) << std::endl; abort(); }
            }
        }
        // one container over ng GPUs (SURVEY.md 8e): every context probes its own range of chunks, the host hands each shard's probe
        // records to the others, every context replays the accept logic and keeps the plaintext of the streams it owns
        std::vector<int> rcs(ng, 0); std::vector<uint64_t> ns(ng, 0);
        auto all = [&](auto fn) {
            std::vector<std::thread> th;
            for (int g = 1; g < ng; g++) th.emplace_back(fn, g);
            fn(0);
            for (auto &t : th) t.join();
            for (int g = 0; g < ng; g++) if (rcs[g] != ATZ_OK) { std::cout << atz_err(ctxs[g], rcs[g]) << std::endl; abort(); }
        };
        all([&](int g) {
            rcs[g] = ng == 1 ? atz_load(ctxs[g], file.data(), file.size()) : atz_attach(ctxs[g], file.data(), file.size());
            if (rcs[g] == ATZ_OK) rcs[g] = atz_scan_shard(ctxs[g], options.chunksize, (uint32_t)g, (uint32_t)ng);
        });
        if (ng > 1) {
            std::vector<std::vector<uint8_t>> blob(ng);
            for (int g = 0; g < ng; g++) {
                uint64_t nb = 0; atz_probe_export(ctxs[g], nullptr, 0, &nb);
                blob[g].resize(nb ? nb : 1);
                rcs[g] = atz_probe_export(ctxs[g], blob[g].data(), nb, &nb); blob[g].resize(nb);
            }
            for (int g = 0; g < ng; g++) for (int h = 0; h < ng; h++) if (h != g && rcs[g] == ATZ_OK) rcs[g] = atz_probe_import(ctxs[g], (uint32_t)h, blob[h].data(), blob[h].size());
        }
        all([&](int g) { if (rcs[g] == ATZ_OK) rcs[g] = atz_scan_finish(ctxs[g], &ns[g]); });
        for (int g = 1; g < ng; g++) if (ns[g] != ns[0]) { std::cout << "error: shards disagree on the stream list" << std::endl; abort(); }
        nstreams = ns[0];
        std::cout << "Total zlib headers found: " << nstreams << std::endl;
        processingState = 1;
        return 0;
    }
    int Phase2() {   // merged into Phase1 by the reference as well (main.cpp:272-285)
        if (processingState != 1) return -10;
        processingState = 2;
        return 0;
    }
    int Phase3() {   // parameter search (findDeflateParams_ALL)
        if (processingState != 2) return -10;
        atz_options o{};
        o.recompTresh = options.recompTresh; o.sizediffTresh = options.sizediffTresh; o.shortcutLength = options.shortcutLength;
        o.mismatchTol = options.mismatchTol; o.bruteforceWindow = options.bruteforceWindow; o.flags = (options.exactRecords ? ATZ_F_EXACT_RECORDS : 0) | (options.strategies ? ATZ_F_STRATEGIES : 0);
        o.flags |= ATZ_F_NESTED_DEPTH(options.nested);
        int ng = (int)ctxs.size();
        std::vector<int> rcs(ng, 0);
        auto work = [&](int g) { rcs[g] = atz_search_shard(ctxs[g], &o, (uint32_t)g, (uint32_t)ng); };
        std::vector<std::thread> th;
        for (int g = 1; g < ng; g++) th.emplace_back(work, g);
        work(0);
        for (auto &t : th) t.join();
        for (int g = 0; g < ng; g++) if (rcs[g] != ATZ_OK) { std::cout << atz_err(ctxs[g], rcs[g]) << std::endl; abort(); }
        // host-side gather of the fixed-size best-candidate records: stream i lives on the context that owns it (atz_get_owners)
        streams.clear();
        std::vector<std::vector<atz_stream>> per(ng, std::vector<atz_stream>(nstreams ? nstreams : 1));
        std::vector<std::vector<uint64_t>> doff(ng); std::vector<std::vector<uint8_t>> dval(ng);
        for (int g = 0; g < ng; g++) {
            atz_get_streams(ctxs[g], per[g].data(), nstreams);
            uint64_t nd = 0; atz_get_diffs(ctxs[g], nullptr, nullptr, 0, &nd);
            doff[g].resize(nd ? nd : 1); dval[g].resize(nd ? nd : 1);
            if (nd) atz_get_diffs(ctxs[g], doff[g].data(), dval[g].data(), nd, &nd);
        }
        owner.assign(nstreams ? nstreams : 1, 0);
        atz_get_owners(ctxs[0], owner.data(), nstreams);
        for (uint64_t i = 0; i < nstreams; i++) {
            int g = (int)owner[i]; const atz_stream &a = per[g][i];
            ATZdata::streamOffset s(a.offset, a.offsetType, a.streamLength, a.inflatedLength);
            s.zlibparams = ATZdata::zlibParamPack(a.clevel, a.window, a.memlevel);
            s.identBytes = a.identBytes; s.firstDiffByte = a.firstDiffByte; s.recomp = a.recomp != 0;
            s.diffByteOffsets.assign(doff[g].begin() + a.diff_index, doff[g].begin() + a.diff_index + a.ndiff);
            s.diffByteVal.assign(dval[g].begin() + a.diff_index, dval[g].begin() + a.diff_index + a.ndiff);
            if (options.png || options.apng) {
                uint64_t np = 0; atz_get_pieces(ctxs[g], i, nullptr, 0, &np);
                s.pieces.resize(np);
                if (np && (atz_get_pieces(ctxs[g], i, s.pieces.data(), np, &np) != ATZ_OK || atz_get_framing(ctxs[g], i, &s.frame) != ATZ_OK)) { std::cout << atz_err(ctxs[g], -1) << std::endl; abort(); }
            }
            streams.push_back(std::move(s));
        }
        // nested streams (--nested): each context lists the ones under the streams it owns; their parent indices are turned into the
        // tree below (kids[i] for top-level stream i, nests[k].kids for nested stream k, in offset order)
        kids.assign(nstreams, {}); nests.clear();
        for (int g = 0; g < ng && options.nested; g++) {
            uint64_t nn = 0; atz_get_nested(ctxs[g], nullptr, 0, &nn);
            std::vector<atz_nested> v(nn ? nn : 1);
            if (nn && atz_get_nested(ctxs[g], v.data(), nn, &nn) != ATZ_OK) { std::cout << atz_err(ctxs[g], -1) << std::endl; abort(); }
            const size_t base = nests.size();
            for (uint64_t j = 0; j < nn; j++) {
                const atz_stream &a = v[j].s;
                Nest n{ATZdata::streamOffset(a.offset, a.offsetType, a.streamLength, a.inflatedLength), g, nstreams + j, {}, {}};
                n.s.zlibparams = ATZdata::zlibParamPack(a.clevel, a.window, a.memlevel);
                n.s.identBytes = a.identBytes; n.s.firstDiffByte = a.firstDiffByte; n.s.recomp = a.recomp != 0;
                n.s.diffByteOffsets.assign(doff[g].begin() + a.diff_index, doff[g].begin() + a.diff_index + a.ndiff);
                n.s.diffByteVal.assign(dval[g].begin() + a.diff_index, dval[g].begin() + a.diff_index + a.ndiff);
                nests.push_back(std::move(n));
                const uint64_t p = v[j].parent;
                if (p < nstreams) kids[p].push_back(base + j);
                else nests[base + (p - nstreams)].kids.push_back(base + j);
            }
        }
        std::cout << std::endl;
        std::cout << "recompressed:" << countRecomp() << "/" << streams.size() << std::endl;
        if (options.nested) {
            uint64_t nr = 0; for (auto &n : nests) nr += n.s.recomp;
            std::cout << "nested recompressed:" << nr << "/" << nests.size() << std::endl;
        }
        processingState = 3;
        return 0;
    }
    int Phase4() {   // ATZ1 writer
        if (processingState != 3) return -10;
        writeATZfile();
        if (options.stats) printStats();
        streams.clear(); streams.shrink_to_fit();
        processingState = 3;
        return 0;
    }

  private:
    std::string infileName, atzfileName, reconfileName;
    ATZdata::programOptions options;
    int processingState = 0;
    uint64_t infileSize = 0, nstreams = 0;
    MappedFile file;
    std::vector<atz_ctx *> ctxs;
    std::vector<uint32_t> owner;   // shard that holds stream i's record and plaintext
    std::vector<ATZdata::streamOffset> streams;
    struct Nest { ATZdata::streamOffset s; int g; uint64_t idx; std::vector<size_t> kids; std::vector<uint8_t> plain; };   // g: context, idx: its atz_get_inflated index
    std::vector<Nest> nests; std::vector<std::vector<size_t>> kids;

    uint64_t countRecomp() { uint64_t n = 0; for (auto &s : streams) if (s.recomp) n++; return n; }

    // ATZ1 layout (main.cpp:775-831): header, per recompressed stream {descriptor, diffs, inflated data}, residue.  A stream split over
    // PNG IDAT chunks (--png) has bit 7 of its window byte set and, behind the diffs, u64 npieces, npieces u32 piece lengths and the
    // (npieces - 1) x 12 framing bytes between the pieces, copied from the input (its CRCs stay exact even where they are wrong).  One
    // split over APNG fdAT chunks (--apng) sets bits 7 and 5, and its framing is 16 bytes per gap (the sequence numbers stay exact too).
    // A stream with recompressed nested streams (--nested) has bit 6 of its window byte set, and its payload P is replaced by u64 nchild,
    // the records of those nchild streams in offset order (the same layout, recursively; never bit 7) and P without their bytes.
    static bool any_recomp(const std::vector<Nest> &ns, const std::vector<size_t> &k) { for (size_t i : k) if (ns[i].s.recomp) return true; return false; }
    void put_payload(std::vector<uint8_t> &out, const uint8_t *P, uint64_t U, const std::vector<size_t> &k) {
        if (!any_recomp(nests, k)) { out.insert(out.end(), P, P + U); return; }
        uint64_t nc = 0; for (size_t i : k) nc += nests[i].s.recomp;
        put8(out, nc);
        for (size_t i : k) {
            const Nest &n = nests[i]; const auto &s = n.s;
            if (!s.recomp) continue;
            put8(out, s.offset); put8(out, s.streamLength); put8(out, s.inflatedLength);
            out.push_back(s.zlibparams.clevel); out.push_back(s.zlibparams.window | (any_recomp(nests, n.kids) ? 0x40 : 0)); out.push_back(s.zlibparams.memlevel);
            const uint64_t nd = s.diffByteOffsets.size();
            put8(out, nd);
            if (nd > 0) {
                put8(out, (uint64_t)s.firstDiffByte);
                for (uint64_t q = 0; q < nd; q++) put8(out, s.diffByteOffsets[q]);
                for (uint64_t q = 0; q < nd; q++) out.push_back(s.diffByteVal[q]);
            }
            put_payload(out, n.plain.data(), s.inflatedLength, n.kids);
        }
        uint64_t at = 0;    // the residue
        for (size_t i : k) if (nests[i].s.recomp) { out.insert(out.end(), P + at, P + nests[i].s.offset); at = nests[i].s.offset + nests[i].s.streamLength; }
        out.insert(out.end(), P + at, P + U);
    }
    void writeATZfile() {
        uint64_t total = 28, nrec = countRecomp();
        for (auto &s : streams) if (s.recomp) total += 35 + (s.diffByteOffsets.empty() ? 0 : 8 + 9 * s.diffByteOffsets.size()) + s.inflatedLength + (s.pieces.empty() ? 0 : 8 + 4 * s.pieces.size() + (uint64_t)s.frame * (s.pieces.size() - 1));
        std::vector<uint8_t> out; out.reserve(total + infileSize);
        out.insert(out.end(), {'A', 'T', 'Z', 1});
        put8(out, 0); put8(out, infileSize); put8(out, nrec);
        // every recompressed stream's plaintext in one gather + one copy per GPU (it has been resident on the device that owns the
        // stream since phase 1) instead of the reference's per-stream re-read and re-inflate (main.cpp:824-828)
        const int ng = (int)ctxs.size();
        std::vector<std::vector<uint64_t>> which(ng); std::vector<uint64_t> paybytes(ng, 0), pay_at(ng, 0);
        for (uint64_t i = 0; i < streams.size(); i++) if (streams[i].recomp) { which[owner[i]].push_back(i); paybytes[owner[i]] += streams[i].inflatedLength; }
        std::vector<std::vector<uint8_t>> payload(ng);
        {
            std::vector<int> rcs(ng, ATZ_OK); std::vector<uint64_t> got(ng, 0);
            auto fetch = [&](int g) {
                payload[g].resize(paybytes[g] ? paybytes[g] : 1);
                if (!which[g].empty()) rcs[g] = atz_get_inflated_list(ctxs[g], which[g].data(), which[g].size(), payload[g].data(), paybytes[g], &got[g]);
            };
            std::vector<std::thread> th;
            for (int g = 1; g < ng; g++) th.emplace_back(fetch, g);
            fetch(0);
            for (auto &t : th) t.join();
            for (int g = 0; g < ng; g++) if (rcs[g] != ATZ_OK || got[g] != (which[g].empty() ? 0 : paybytes[g])) { std::cout << atz_err(ctxs[g], rcs[g]) << std::endl; abort(); }
            // the plaintext of the recompressed nested streams, from the context that found them
            for (int g = 0; g < ng && !nests.empty(); g++) {
                std::vector<uint64_t> idx; std::vector<size_t> at; uint64_t tot = 0, got2 = 0;
                for (size_t i = 0; i < nests.size(); i++) if (nests[i].g == g && nests[i].s.recomp) { idx.push_back(nests[i].idx); at.push_back(i); tot += nests[i].s.inflatedLength; }
                if (idx.empty()) continue;
                std::vector<uint8_t> buf(tot ? tot : 1);
                const int rc = atz_get_inflated_list(ctxs[g], idx.data(), idx.size(), buf.data(), tot, &got2);
                if (rc != ATZ_OK || got2 != tot) { std::cout << atz_err(ctxs[g], rc) << std::endl; abort(); }
                uint64_t o = 0;
                for (size_t i : at) { nests[i].plain.assign(buf.begin() + o, buf.begin() + o + nests[i].s.inflatedLength); o += nests[i].s.inflatedLength; }
            }
        }
        for (uint64_t i = 0; i < streams.size(); i++) {
            auto &s = streams[i];
            if (!s.recomp) continue;
            put8(out, s.offset); put8(out, s.streamLength); put8(out, s.inflatedLength);
            out.push_back(s.zlibparams.clevel); out.push_back(s.zlibparams.window | (s.pieces.empty() ? 0 : s.frame == 16 ? 0xa0 : 0x80) | (any_recomp(nests, kids[i]) ? 0x40 : 0)); out.push_back(s.zlibparams.memlevel);
            uint64_t nd = s.diffByteOffsets.size();
            put8(out, nd);
            if (nd > 0) {
                put8(out, (uint64_t)s.firstDiffByte);
                for (uint64_t k = 0; k < nd; k++) put8(out, s.diffByteOffsets[k]);
                for (uint64_t k = 0; k < nd; k++) out.push_back(s.diffByteVal[k]);
            }
            if (!s.pieces.empty()) {
                put8(out, s.pieces.size());
                for (uint32_t l : s.pieces) for (int b = 0; b < 4; b++) out.push_back((uint8_t)(l >> (8 * b)));
                uint64_t at = s.offset;
                for (size_t k = 0; k + 1 < s.pieces.size(); k++) { at += s.pieces[k]; out.insert(out.end(), file.begin() + at, file.begin() + at + s.frame); at += s.frame; }
            }
            const uint32_t g = owner[i];
            put_payload(out, payload[g].data() + pay_at[g], s.inflatedLength, kids[i]); pay_at[g] += s.inflatedLength;
        }
        uint64_t lastos = 0, lastlen = 0;   // residue: gaps, non-recompressed streams, tail (main.cpp:784-796)
        for (auto &s : streams) {
            if ((lastos + lastlen) != s.offset) out.insert(out.end(), file.begin() + (lastos + lastlen), file.begin() + s.offset);
            if (!s.recomp) out.insert(out.end(), file.begin() + s.offset, file.begin() + s.offset + s.spanLength());
            lastos = s.offset; lastlen = s.spanLength();
        }
        if ((lastos + lastlen) < infileSize) out.insert(out.end(), file.begin() + (lastos + lastlen), file.end());
        uint64_t atzlen = out.size();
        for (int i = 0; i < 8; i++) out[4 + i] = (uint8_t)(atzlen >> (8 * i));
        std::ofstream outfile(atzfileName, std::ios::out | std::ios::binary | std::ios::trunc);
        if (!outfile.is_open()) { std::cout << "error: open file for output failed!" << std::endl; abort(); }
        outfile.write(reinterpret_cast<const char *>(out.data()), (std::streamsize)out.size());
        std::cout << "Total bytes written: " << atzlen << std::endl;
    }
    void printStats() {
        for (size_t g = 0; g < ctxs.size(); g++) {
            atz_stats st; atz_get_stats(ctxs[g], &st);
            std::cerr << "[gpu " << g << "] candidates " << st.n_candidates << " streams " << st.n_streams << " ref_trials " << st.ref_trials << " gpu_trials " << st.gpu_trials
                      << " | ms: h2d " << st.ms_h2d << " scan " << st.ms_scan << " probe " << st.ms_inflate_probe << " inflate " << st.ms_inflate << " chains " << st.ms_chains
                      << " trials " << st.ms_trials << " diff " << st.ms_diff << " d2h " << st.ms_d2h << " | algo_bytes " << st.algo_bytes << " launches " << st.kernel_launches << std::endl;
        }
    }
};

// ---------------------------------------------------------------------------------------------
static bool g_print_stats = false;   // --stats, for the reconstruct path too

class ATZreconstructor {
  public:
    ATZreconstructor(std::string atz, std::string rec, int device = 0) : atzfileName(atz), reconfileName(rec), dev(device) {}
    int reconstructATZ(const uint64_t /*chunksize*/) {
        uint64_t origlen = 0, nstrms = 0, atzfileSize = 0;
        std::cout << "reconstructing from " << atzfileName << std::endl;
        std::vector<uint8_t> atz;
        if (parseATZheader(atz, origlen, nstrms) != 0) return -1;
        atzfileSize = atz.size();
        std::cout << "ATZ file size: " << atzfileSize << std::endl;
        std::cout << "Original file size: " << origlen << std::endl;
        std::ofstream recfile(reconfileName, std::ios::out | std::ios::binary | std::ios::trunc);
        auto invalid = [](const char *what) { std::cout << "Invalid file: " << what << std::endl; return -1; };
        if (nstrms == 0) {   // main.cpp:941-948
            if (origlen > atzfileSize - 28) return invalid("original length exceeds the ATZ file");
            recfile.write(reinterpret_cast<const char *>(atz.data() + 28), (std::streamsize)origlen);
            return 0;
        }
        if (nstrms > (atzfileSize - 28) / 35) return invalid("stream count exceeds the ATZ file");
        std::vector<ATZdata::streamOffset> list;
        uint64_t residueos = readStreamdesc_ALL(atz, list, nstrms, origlen);
        // every stream's doDeflate (main.cpp:914, 976-1003) in batched kernel launches
        atz_ctx *ctx = nullptr;
        if (atz_ctx_create(dev, &ctx) != ATZ_OK) { std::cout << "error: no usable CUDA device (antiz_b200 has no CPU path)" << std::endl; std::exit(1); }
        const uint64_t n = list.size();
        {   // the reference reads through an ifstream, which just comes up short on a damaged file; this reader indexes a buffer, so every
            // offset the descriptors imply is checked first: streams ascending and disjoint, inside the original, residue inside the ATZ file
            uint64_t end = 0, gaps = 0;
            for (uint64_t j = 0; j < n; j++) {
                const auto &s = list[j];
                if (s.offset < end || s.offset > origlen || s.spanLength() > origlen - s.offset) return invalid("stream descriptors out of order or outside the original file");
                gaps += s.offset - end; end = s.offset + s.spanLength();
                if (s.streamLength >= 0xffff0000ull || s.inflatedLength >= 0xffffff00ull) return invalid("stream too large");
                if ((s.zlibparams.clevel & 15) > 9 || (s.zlibparams.clevel >> 4) > 4 || s.zlibparams.window < 9 || s.zlibparams.window > 15 || s.zlibparams.memlevel < 1 || s.zlibparams.memlevel > 9) return invalid("bad zlib parameters");
            }
            gaps += origlen - end;
            if (residueos > atzfileSize || gaps > atzfileSize - residueos) return invalid("residue exceeds the ATZ file");
        }
        if (!nodes.empty() && rebuildNested(ctx, atz, list) != ATZ_OK) abort();
        std::vector<uint64_t> in_off(n), in_len(n), out_off(n), out_cap(n), out_len(n);
        std::vector<uint8_t> cl(n), wb(n), ml(n);
        uint64_t oo = 0;
        for (uint64_t j = 0; j < n; j++) {
            in_off[j] = list[j].atzInfos; in_len[j] = list[j].inflatedLength;
            out_off[j] = oo; out_cap[j] = list[j].streamLength + 65535; oo += out_cap[j];   // same capacity as main.cpp:910
            cl[j] = list[j].zlibparams.clevel; wb[j] = list[j].zlibparams.window; ml[j] = list[j].zlibparams.memlevel;
        }
        std::vector<uint8_t> comp(oo ? oo : 1);
        int rc = atz_deflate_batch(ctx, atz.data(), in_off.data(), in_len.data(), cl.data(), wb.data(), ml.data(), n, comp.data(), out_off.data(), out_cap.data(), out_len.data());
        if (rc != ATZ_OK) { std::cout << "deflate() failed with exit code:" << rc << " " << atz_last_error(ctx) << std::endl; abort(); }
        if (g_print_stats) {
            atz_stats st; atz_get_stats(ctx, &st);
            std::cerr << "[gpu reconstruct] streams " << n << " | ms: h2d " << st.ms_h2d << " chains " << st.ms_chains << " rows " << st.ms_rows << " deflate " << st.ms_trials
                      << " d2h " << st.ms_d2h << " | launches " << st.kernel_launches << std::endl;
        }
        atz_ctx_destroy(ctx);
        uint64_t gapsum = 0, lastos = 0, lastlen = 0;
        for (uint64_t j = 0; j < n; j++) {
            auto &s = list[j];
            if ((lastos + lastlen) != s.offset) {
                uint64_t gap = s.offset - (lastos + lastlen);
                recfile.write(reinterpret_cast<const char *>(atz.data() + residueos + gapsum), (std::streamsize)gap);
                gapsum += gap;
            }
            uint8_t *cb = comp.data() + out_off[j];
            if (s.firstDiffByte >= 0) {   // patch list (main.cpp:916-926)
                uint64_t sum = 0;
                for (uint64_t i = 0; i < s.diffByteOffsets.size(); i++) {
                    uint64_t pos = (uint64_t)s.firstDiffByte + s.diffByteOffsets[i] + sum;
                    if (pos < out_cap[j]) cb[pos] = s.diffByteVal[i];
                    sum += s.diffByteOffsets[i];
                }
            }
            if (s.pieces.empty()) recfile.write(reinterpret_cast<const char *>(cb), (std::streamsize)s.streamLength);
            else {   // piece 1, framing 1, piece 2, ...
                uint64_t at = 0;
                for (size_t k = 0; k < s.pieces.size(); k++) {
                    recfile.write(reinterpret_cast<const char *>(cb + at), (std::streamsize)s.pieces[k]); at += s.pieces[k];
                    if (k + 1 < s.pieces.size()) recfile.write(reinterpret_cast<const char *>(atz.data() + s.gapsAt + s.frame * k), s.frame);
                }
            }
            lastos = s.offset; lastlen = s.spanLength();
        }
        if ((lastos + lastlen) < origlen) recfile.write(reinterpret_cast<const char *>(atz.data() + residueos + gapsum), (std::streamsize)(origlen - (lastos + lastlen)));
        recfile.close();
        return 0;
    }

  private:
    std::string atzfileName, reconfileName; int dev;
    struct Tree { std::vector<size_t> kids; uint64_t residueAt = 0; };   // a record's nested streams (indices into nodes) and where its residue starts
    struct Node { ATZdata::streamOffset s; Tree t; int depth; };
    std::vector<Tree> tops; std::vector<Node> nodes;
    int parseATZheader(std::vector<uint8_t> &atz, uint64_t &origlen, uint64_t &nstrms) {   // main.cpp:1011-1030
        uint64_t infileSize = 0;
        if (getFilesize(atzfileName, infileSize) != 0) return -1;
        read_file(atzfileName, atz);
        if (atz.size() < 4 || atz[0] != 'A' || atz[1] != 'T' || atz[2] != 'Z' || atz[3] != 1) { std::cout << "Invalid file: ATZ1 header not found" << std::endl; return -2; }
        if (atz.size() < 28 || get8(&atz[4]) != infileSize) { std::cout << "Invalid file: ATZ file size mismatch" << std::endl; return -3; }
        origlen = get8(&atz[12]); nstrms = get8(&atz[20]);
        return 0;
    }
    uint64_t readStreamdesc_ALL(const std::vector<uint8_t> &atz, std::vector<ATZdata::streamOffset> &list, uint64_t nstrms, uint64_t origlen) {   // main.cpp:1031-1063
        uint64_t lastos = 28;
        tops.assign(nstrms, Tree());
        for (uint64_t j = 0; j < nstrms; j++) {
            list.push_back(ATZdata::streamOffset(0, -1, 0, 0));
            lastos = readRecord(atz, lastos, origlen, 0, list[j], tops[j]);
        }
        return lastos;
    }
    // One record at `lastos`: descriptor, diffs, (window bit 7, --png; with bit 5, --apng) the piece table and framing bytes, then the payload or (bit 6,
    // --nested) u64 nchild, the nested records and the residue.  depth 0 = a top-level record.  Returns the end of the record.
    uint64_t readRecord(const std::vector<uint8_t> &atz, uint64_t lastos, uint64_t origlen, int depth, ATZdata::streamOffset &s, Tree &t) {
        auto need = [&](uint64_t end) { if (end > atz.size()) { std::cout << "Invalid file: truncated stream description" << std::endl; std::exit(1); } };
        auto invalid = [](const char *what) { std::cout << "Invalid file: " << what << std::endl; std::exit(1); };
        need(lastos + 35);
        s = ATZdata::streamOffset(get8(&atz[lastos]), -1, get8(&atz[lastos + 8]), get8(&atz[lastos + 16]));
        s.zlibparams.clevel = atz[lastos + 24]; s.zlibparams.window = atz[lastos + 25]; s.zlibparams.memlevel = atz[lastos + 26];
        uint64_t diffbytes = get8(&atz[lastos + 27]);
        if (diffbytes > 0) {
            if (diffbytes > (atz.size() - lastos) / 9) need(atz.size() + 1);   // (the multiplication below cannot wrap)
            need(lastos + 43 + diffbytes * 9);
            s.firstDiffByte = (int_fast64_t)get8(&atz[lastos + 35]);
            for (uint64_t i = 0; i < diffbytes; i++) {
                s.diffByteOffsets.push_back(get8(&atz[43 + 8 * i + lastos]));
                s.diffByteVal.push_back(atz[43 + diffbytes * 8 + i + lastos]);
            }
            s.atzInfos = 43 + diffbytes * 9 + lastos;
        } else {
            s.firstDiffByte = -1;
            s.atzInfos = 35 + lastos;
        }
        const bool has_nested = s.zlibparams.window & 0x40;
        s.zlibparams.window &= 0xbf;
        if (depth > 0) {
            if (s.zlibparams.window & 0x80) invalid("a nested stream cannot be split over IDAT chunks");
            if (s.zlibparams.window & 0x20) invalid("a nested stream cannot be split over fdAT chunks");
            if ((s.zlibparams.clevel & 15) > 9 || (s.zlibparams.clevel >> 4) > 4 || s.zlibparams.window < 9 || s.zlibparams.window > 15 || s.zlibparams.memlevel < 1 || s.zlibparams.memlevel > 9) invalid("bad zlib parameters");
            if (s.streamLength >= 0xffff0000ull || s.inflatedLength >= 0xffffff00ull) invalid("stream too large");
        }
        if ((s.zlibparams.window & 0xa0) == 0x20) invalid("fdAT framing on a stream that is not split");
        if (s.zlibparams.window & 0x80) {   // split over PNG IDAT chunks (--png) or, bit 5, APNG fdAT chunks (--apng): piece table and framing bytes, checked before any GPU work
            if (s.zlibparams.window & 0x20) s.frame = 16;
            s.zlibparams.window &= 0x5f;
            if (s.zlibparams.window < 9 || s.zlibparams.window > 15) invalid("bad window of a split stream");
            need(s.atzInfos + 8);
            const uint64_t np = get8(&atz[s.atzInfos]);
            if (np < 2) invalid("a split stream needs at least 2 pieces");
            if (np > (atz.size() - s.atzInfos - 8) / (4 + s.frame) + 1) need(atz.size() + 1);   // (the sizes below cannot wrap)
            need(s.atzInfos + 8 + 4 * np + s.frame * (np - 1));
            uint64_t sum = 0;
            for (uint64_t k = 0; k < np; k++) { uint32_t l; std::memcpy(&l, &atz[s.atzInfos + 8 + 4 * k], 4); s.pieces.push_back(l); sum += l; }
            if (sum != s.streamLength) invalid("piece lengths of a split stream do not sum to its length");
            if (s.offset > origlen || s.spanLength() > origlen - s.offset) invalid("split stream outside the original file");
            s.gapsAt = s.atzInfos + 8 + 4 * np;
            s.atzInfos += 8 + 4 * np + s.frame * (np - 1);
        }
        if (s.inflatedLength > atz.size()) need(atz.size() + 1);
        if (!has_nested) {
            lastos = s.atzInfos + s.inflatedLength;
            need(lastos);
            return lastos;
        }
        // nested records: ascending, disjoint, inside [0, U) of this plaintext; the residue is U minus their compressed bytes
        if (depth >= 8) invalid("streams nested deeper than 8 levels");
        need(s.atzInfos + 8);
        const uint64_t nchild = get8(&atz[s.atzInfos]);
        if (nchild == 0) invalid("a stream marked as holding nested streams has none");
        if (nchild > (atz.size() - s.atzInfos - 8) / 35) need(atz.size() + 1);
        uint64_t pos = s.atzInfos + 8, end = 0, sumc = 0;
        for (uint64_t k = 0; k < nchild; k++) {
            ATZdata::streamOffset c(0, -1, 0, 0); Tree ct;
            pos = readRecord(atz, pos, origlen, depth + 1, c, ct);
            if (c.offset < end || c.offset >= s.inflatedLength || c.streamLength > s.inflatedLength - c.offset) invalid("nested streams out of order or outside their parent's plaintext");
            end = c.offset + c.streamLength; sumc += c.streamLength;
            nodes.push_back(Node{std::move(c), std::move(ct), depth + 1});
            t.kids.push_back(nodes.size() - 1);
        }
        t.residueAt = pos;
        lastos = pos + (s.inflatedLength - sumc);
        need(lastos);
        return lastos;
    }
    // --nested: the plaintext of every stream with nested streams, deepest level first: the level's streams are deflated in one batch and
    // patched, then each parent's plaintext is put together from its residue and its children's bytes and appended to `atz`, where the
    // parent's atzInfos then points
    int rebuildNested(atz_ctx *ctx, std::vector<uint8_t> &atz, std::vector<ATZdata::streamOffset> &list) {
        int maxd = 0;
        for (const Node &n : nodes) maxd = std::max(maxd, n.depth);
        std::vector<std::vector<uint8_t>> comp(nodes.size());
        for (int d = maxd; d >= 1; d--) {
            std::vector<size_t> lv;
            for (size_t i = 0; i < nodes.size(); i++) if (nodes[i].depth == d) lv.push_back(i);
            const uint64_t n = lv.size();
            std::vector<uint64_t> in_off(n), in_len(n), out_off(n), out_cap(n), out_len(n);
            std::vector<uint8_t> cl(n), wb(n), ml(n);
            uint64_t oo = 0;
            for (uint64_t j = 0; j < n; j++) {
                const auto &s = nodes[lv[j]].s;
                in_off[j] = s.atzInfos; in_len[j] = s.inflatedLength;
                out_off[j] = oo; out_cap[j] = s.streamLength + 65535; oo += out_cap[j];
                cl[j] = s.zlibparams.clevel; wb[j] = s.zlibparams.window; ml[j] = s.zlibparams.memlevel;
            }
            std::vector<uint8_t> out(oo ? oo : 1);
            const int rc = atz_deflate_batch(ctx, atz.data(), in_off.data(), in_len.data(), cl.data(), wb.data(), ml.data(), n, out.data(), out_off.data(), out_cap.data(), out_len.data());
            if (rc != ATZ_OK) { std::cout << "deflate() failed with exit code:" << rc << " " << atz_last_error(ctx) << std::endl; return rc; }
            for (uint64_t j = 0; j < n; j++) {
                const auto &s = nodes[lv[j]].s;
                uint8_t *cb = out.data() + out_off[j];
                if (s.firstDiffByte >= 0) {
                    uint64_t sum = 0;
                    for (uint64_t i = 0; i < s.diffByteOffsets.size(); i++) {
                        const uint64_t pos = (uint64_t)s.firstDiffByte + s.diffByteOffsets[i] + sum;
                        if (pos < out_cap[j]) cb[pos] = s.diffByteVal[i];
                        sum += s.diffByteOffsets[i];
                    }
                }
                comp[lv[j]].assign(cb, cb + s.streamLength);
            }
            auto splice = [&](ATZdata::streamOffset &s, const Tree &t) {
                std::vector<uint8_t> P; P.reserve(s.inflatedLength);
                uint64_t res = t.residueAt, at = 0;
                for (size_t k : t.kids) {
                    const auto &c = nodes[k].s;
                    P.insert(P.end(), atz.begin() + res, atz.begin() + res + (c.offset - at)); res += c.offset - at;
                    P.insert(P.end(), comp[k].begin(), comp[k].end()); at = c.offset + c.streamLength;
                }
                P.insert(P.end(), atz.begin() + res, atz.begin() + res + (s.inflatedLength - at));
                s.atzInfos = atz.size();
                atz.insert(atz.end(), P.begin(), P.end());
            };
            for (Node &p : nodes) if (p.depth == d - 1 && !p.t.kids.empty()) splice(p.s, p.t);
            if (d == 1) for (size_t j = 0; j < list.size(); j++) if (!tops[j].kids.empty()) splice(list[j], tops[j]);
        }
        return ATZ_OK;
    }
};

// ---------------------------------------------------------------------------------------------
// ---- command line: the reference's TCLAP front end (main.cpp:1075-1143) restated ----
// The usage / help / error texts, their layout (75 columns, the continuation indent of the usage line, errors and the brief
// usage on stderr) and the exit codes are the reference's; tests/test_cli.py compares them with the reference binary's.
struct CliArg { const char *flag, *name, *type; bool required; const char *desc; };   // flag: "" = none; type: nullptr = switch
static const CliArg kArgs[] = {
    {"", "brute-window", nullptr, false, "Bruteforce deflate window size if there is a chance that recompression could be improved by it. This can have a major performance penalty. Default: disabled"},
    {"", "notest", nullptr, false, "Skip comparing the reconstructed file to the original at the end. This is not recommended, as AntiZ is still experimental software and my contain bugs that corrupt data."},
    {"r", "reconstruct", nullptr, false, "Assume the input file is an ATZ file and attempt to reconstruct the original file from it"},
    {"", "chunksize", "integer", false, "Size of the memory buffer in bytes for chunked disk IO. This contorls memory usage to some extent, but memory usage control is not fully implemented yet. Smaller values result in more disk IO operations. Default: 524288"},
    {"", "mismatch-tol", "integer", false, "Mismatch tolerance in bytes. If a set of parameters are found that give at most this many mismatches, then accept them and stop looking for a better set of parameters. Increasing this improves speed at the cost of more ATZ file overhead that may hurt compression. Default: 2  Maximum: 65535"},
    {"", "shortcut-len", "integer", false, "Length of the shortcut in bytes. If a stream is longer than the shortcut, then stop compression after <shortcut> compressed bytes have been obtained and compare this portion to the original. If this comparison yields more than recompTresh mismatches, then do not compress the entire stream. Lowering this improves speed, but it must be significantly greater than recompTresh or the speed benefit will decrease. Default: 512  Maximum: 65535"},
    {"", "sizediff-tresh", "integer", false, "Size difference treshold in bytes. If the size difference between a recompressed stream and the original is more than the treshold then do not even compare them. Increasing this treshold increases the chance that a stream will be compared to the original. The cost of comparing is relatively low, so setting this equal to the recompression treshold should be fine. Default: 128  Maximum: 65535"},
    {"", "recomp-tresh", "integer", false, "Recompression treshold in bytes. Streams are only recompressed if the best match differs from the original in at most recompTresh bytes. Increasing this treshold may allow more streams to be recompressed, but may increase ATZ file overhead and make it harder to compress. Default: 128  Maximum: 65535"},
    {"o", "output", "string", false, "Output file name"},
    {"i", "input", "string", true, "Input file name"},
    {"-", "ignore_rest", nullptr, false, "Ignores the rest of the labeled arguments following this flag."},
    {"", "version", nullptr, false, "Displays version information and exits."},
    {"h", "help", nullptr, false, "Displays usage information and exits."},
};
static const CliArg kExtArgs[] = {   // antiz_b200 only: listed after the reference's help text, not in its usage line
    {"", "gpus", "integer", false, "Number of GPUs to shard the stream x parameter search over. Default: 1"},
    {"", "device", "integer", false, "First CUDA device ordinal. Default: 0"},
    {"", "exact-records", nullptr, false, "Disable the early cut of hopeless trials (the per-stream records of streams that are not recompressed stay exact; the ATZ file is the same either way)"},
    {"", "stats", nullptr, false, "Print per-phase timings to stderr"},
    {"", "strategies", nullptr, false, "For streams that no plain parameter set reproduces, also try zlib's other strategies (Z_FILTERED, Z_FIXED, Z_RLE, Z_HUFFMAN_ONLY). More streams are recompressed, but the ATZ file then differs from the reference's and only this program can reconstruct from it. Default: disabled"},
    {"", "small-windows", nullptr, false, "Also look for zlib streams with 256- and 512-byte windows (header bytes 0x08 and 0x18). More streams are found and recompressed, so the ATZ file differs from the reference's, but the reference can still reconstruct from it. Default: disabled"},
    {"", "png", nullptr, false, "Also find zlib streams that PNG files split over consecutive IDAT chunks, and recompress them with the chunk framing between the pieces stored verbatim. The ATZ file then differs from the reference's and only this program can reconstruct from it. Default: disabled"},
    {"", "nested", "integer", false, "Also recompress zlib streams found inside the decompressed data of recompressed streams, down to this many levels (0-8). The ATZ file then differs from the reference's and only this program can reconstruct from it. Default: 0"},
    {"", "apng", nullptr, false, "Also find zlib streams that animated PNG files split over consecutive fdAT chunks, and recompress them with the chunk framing and sequence numbers between the pieces stored verbatim. Does not imply --png, which the default image needs. The ATZ file then differs from the reference's and only this program can reconstruct from it. Default: disabled"},
};
static std::string cli_short_id(const CliArg &a) {
    std::string id = a.flag[0] ? std::string("-") + a.flag : std::string("--") + a.name;
    if (a.type) id += std::string(" <") + a.type + ">";
    return a.required ? id : "[" + id + "]";
}
static std::string cli_long_id(const CliArg &a) {
    const std::string v = a.type ? std::string(" <") + a.type + ">" : "";
    std::string id = a.flag[0] ? std::string("-") + a.flag + v + ",  " : "";
    return id + "--" + a.name + v;
}
static std::string cli_err_id(const CliArg &a) { return (a.flag[0] ? std::string("-") + a.flag + " " : std::string()) + "(--" + a.name + ")"; }
// Word wrap the way the reference's help is laid out: lines of at most `width` columns including the indent, broken behind the
// last space, comma or bar that fits (mid-word if there is none), continuation lines indented by `more` extra columns and never
// starting with a space.
static void wrap_print(std::ostream &os, const std::string &s, int width, int indent, int more) {
    const int len = (int)s.size();
    if (len + indent <= width) { os << std::string(indent, ' ') << s << std::endl; return; }
    int room = width - indent, at = 0;
    while (at < len) {
        int take = std::min(len - at, room);
        if (take == room) {
            int cut = take;
            while (cut >= 0 && s[at + cut] != ' ' && s[at + cut] != ',' && s[at + cut] != '|') cut--;
            if (cut > 0) take = cut;
        }
        for (int i = 0; i < take; i++) if (s[at + i] == '\n') { take = i + 1; break; }
        os << std::string(indent, ' ');
        if (at == 0) { indent += more; room -= more; }
        os << s.substr(at, take) << std::endl;
        at += take;
        while (at < len && s[at] == ' ') at++;
    }
}
static void short_usage(std::ostream &os, const char *argv0) {
    std::string s = std::string(argv0) + " ";
    for (const CliArg &a : kArgs) s += " " + cli_short_id(a);
    wrap_print(os, s, 75, 3, std::min<int>((int)std::strlen(argv0) + 2, 75 / 2));
}
static void usage(const char *argv0) {
    std::cout << std::endl << "USAGE: " << std::endl << std::endl;
    short_usage(std::cout, argv0);
    std::cout << std::endl << std::endl << "Where: " << std::endl << std::endl;
    for (const CliArg &a : kArgs) {
        wrap_print(std::cout, cli_long_id(a), 75, 3, 3);
        wrap_print(std::cout, std::string(a.required ? "(required)  " : "") + a.desc, 75, 5, 0);
        std::cout << std::endl;
    }
    std::cout << std::endl;
    wrap_print(std::cout, "Visit https://github.com/Diazonium/AntiZ for source code and support.", 75, 3, 0);
    std::cout << std::endl;
    std::cout << "antiz_b200 extensions: " << std::endl << std::endl;
    for (const CliArg &a : kExtArgs) {
        wrap_print(std::cout, cli_long_id(a), 75, 3, 3);
        wrap_print(std::cout, a.desc, 75, 5, 0);
        std::cout << std::endl;
    }
}
[[noreturn]] static void parse_error(const char *argv0, const std::string &msg, const std::string &arg) {
    std::cerr << "PARSE ERROR: " << (arg.empty() ? std::string(" ") : "Argument: " + arg) << std::endl << "             " << msg << std::endl << std::endl;
    std::cerr << "Brief USAGE: " << std::endl;
    short_usage(std::cerr, argv0);
    std::cerr << std::endl << "For complete USAGE and HELP type: " << std::endl << "   " << argv0 << " --help" << std::endl << std::endl;
    std::exit(1);
}

static void parseCLI(int argc, char *argv[], std::string &infile_name, std::string &atzfile_name, std::string &reconfile_name, ATZdata::programOptions &options) {
    std::string in, out; bool in_set = false, out_set = false;
    std::vector<const CliArg *> seen;
    auto find = [&](const std::string &tok) -> const CliArg * {
        for (const CliArg &a : kArgs) if ((a.flag[0] && tok == std::string("-") + a.flag) || tok == std::string("--") + a.name) return &a;
        for (const CliArg &a : kExtArgs) if (tok == std::string("--") + a.name) return &a;
        return nullptr;
    };
    for (int i = 1; i < argc; i++) {
        const std::string tok = argv[i];
        const CliArg *a = find(tok);
        if (!a) parse_error(argv[0], "Couldn't find match for argument", tok);
        const std::string n = a->name;
        if (n == "ignore_rest") break;   // the rest is left unread, as the reference leaves it
        if (std::find(seen.begin(), seen.end(), a) != seen.end()) parse_error(argv[0], "Argument already set!", cli_err_id(*a));
        seen.push_back(a);
        std::string v;
        if (a->type) {
            if (i + 1 >= argc) parse_error(argv[0], "Missing a value for this argument!", cli_err_id(*a));
            v = argv[++i];
        }
        uint64_t x = 0;
        if (a->type && std::string(a->type) == "integer") {
            char *end = nullptr;
            x = std::strtoull(v.c_str(), &end, 10);
            if (v.empty() || end == v.c_str() || *end) parse_error(argv[0], "Couldn't read argument value from string '" + v + "'", cli_err_id(*a));
        }
        if (n == "input") { in = v; in_set = true; }
        else if (n == "output") { out = v; out_set = true; }
        else if (n == "recomp-tresh") options.recompTresh = x;
        else if (n == "sizediff-tresh") options.sizediffTresh = x;
        else if (n == "shortcut-len") options.shortcutLength = x;
        else if (n == "mismatch-tol") options.mismatchTol = x;
        else if (n == "chunksize") options.chunksize = x;
        else if (n == "reconstruct") options.recon = true;
        else if (n == "notest") options.notest = true;
        else if (n == "brute-window") options.bruteforceWindow = true;
        else if (n == "gpus") options.gpus = (int)x;
        else if (n == "device") options.device = (int)x;
        else if (n == "exact-records") options.exactRecords = true;
        else if (n == "stats") { options.stats = true; g_print_stats = true; }
        else if (n == "strategies") options.strategies = true;
        else if (n == "small-windows") options.smallWindows = true;
        else if (n == "png") options.png = true;
        else if (n == "apng") options.apng = true;
        else if (n == "nested") options.nested = (int)std::min<uint64_t>(x, 9);
        else if (n == "help") { usage(argv[0]); std::exit(0); }
        else if (n == "version") { std::cout << std::endl << argv[0] << "  version: " << antiz_ver << std::endl << std::endl; std::exit(0); }
    }
    if (!in_set) parse_error(argv[0], "Required argument missing: input", "");
    if (options.chunksize < 2) parse_error(argv[0], "chunksize must be at least 2", "(--chunksize)");
    if (options.nested > 8) parse_error(argv[0], "nested depth must be at most 8", "(--nested)");
    std::cout << "Input file: " << in << std::endl;
    if (options.recon) {   // main.cpp:1118-1127
        std::cout << "assuming input file is an ATZ file, attempting to reconstruct" << std::endl;
        atzfile_name = in;
        reconfile_name = out_set ? out : atzfile_name + ".rec";
        std::cout << "overwriting " << reconfile_name << " if present" << std::endl;
    } else {               // main.cpp:1128-1139
        infile_name = in;
        atzfile_name = out_set ? out : infile_name + ".atz";
        reconfile_name = infile_name + ".rec";
        std::cout << "overwriting " << atzfile_name << " and " << reconfile_name << " if present" << std::endl;
    }
}

static bool test_f2f(const std::string &a, const std::string &b) {   // main.cpp:1145-1171
    std::vector<uint8_t> x, y;
    if (!read_file(a, x) || !read_file(b, y)) return false;
    return x == y;
}
static int testATZfile(const std::string &infileName, const std::string &atzfileName, const std::string &reconfileName, uint64_t chunksize, int dev) {   // main.cpp:1173-1203
    uint64_t infileSize = 0, recfileSize = 0;
    ATZreconstructor reconATZ(atzfileName, reconfileName, dev);
    if (reconATZ.reconstructATZ(chunksize) != 0) { std::cerr << "Error Encountered: testATZFile() : Reconstruction Failed" << std::endl; std::exit(1); }
    std::cout << "Testing...";
    getFilesize(infileName, infileSize); getFilesize(reconfileName, recfileSize);
    if (infileSize != recfileSize) { std::cout << "error: size mismatch"; return -1; }
    if (!test_f2f(infileName, reconfileName)) { std::cout << "error: byte mismatch"; return -2; }
    std::cout << "OK! Restoration is bit by bit identical" << std::endl;
    if (remove(reconfileName.c_str()) != 0) { std::cout << "error: cannot delete recfile"; return -3; }
    return 0;
}

int main(int argc, char *argv[]) {
    std::cout << "AntiZ " << antiz_ver << std::endl;
    std::string infile_name, atzfile_name, reconfile_name;
    ATZdata::programOptions options;
    parseCLI(argc, argv, infile_name, atzfile_name, reconfile_name, options);
    if (!options.recon) {
        Timer t;
        ATZcreator createATZ(infile_name, atzfile_name, reconfile_name, options);
        if (createATZ.Phase1() != 0) return -1;
        const double w1 = t.ms();
        if (createATZ.Phase2() != 0) return -1;
        if (createATZ.Phase3() != 0) return -1;
        const double w3 = t.ms();
        if (createATZ.Phase4() != 0) return -1;
        if (options.stats) std::cerr << "[host] wall ms: phase 1 (read, context, scan) " << w1 << " | phase 3 (search) " << w3 - w1 << " | phase 4 (payload, write) " << t.ms() - w3
                                     << " | phases 1-4 " << t.ms() << std::endl;
        if (!options.notest) {
            if (testATZfile(infile_name, atzfile_name, reconfile_name, options.chunksize, options.device) != 0) return -1;
        }
    } else {
        ATZreconstructor reconATZ(atzfile_name, reconfile_name, options.device);
        if (reconATZ.reconstructATZ(options.chunksize) != 0) return -1;
    }
    return 0;
}

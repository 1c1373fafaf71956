// Host-side mirror of the reference's public records (reference: /root/reference/ATZData.h:7-88).
// Same namespace, type and field names, defaults and meaning, so code written against the reference's
// ATZData.h compiles against this one; the layout is this project's own (fields it never used are kept
// only for source compatibility).  `AtzData.h` (the spelling main.cpp:1 includes) forwards here.
#ifndef ANTIZ_B200_ATZDATA_H
#define ANTIZ_B200_ATZDATA_H
#include <cstdint>
#include <vector>

namespace ATZdata {

struct programOptions {
    uint_fast16_t recompTresh = 128;     // recompress only if best match differs in <= recompTresh bytes
    uint_fast16_t sizediffTresh = 128;   // compare only if |C' - C| <= sizediffTresh
    uint_fast16_t shortcutLength = 512;  // compare the first shortcutLength output bytes before finishing a trial
    uint_fast16_t mismatchTol = 2;       // <= mismatchTol mismatches counts as a full match
    bool bruteforceWindow = false;
    uint64_t chunksize = 524288;
    bool shortcutEnabled = true;         // debug knob of the reference; always on here
    int_fast64_t concentrate = -1;       // debug knob of the reference; unused
    bool recon = false;
    bool notest = false;
    // antiz_b200 extensions (not in the reference)
    int gpus = 1;                        // shard the stream x parameter grid over this many GPUs
    int device = 0;                      // first device ordinal
    bool exactRecords = false;           // ATZ_F_EXACT_RECORDS
    bool stats = false;                  // print per-phase timings
    bool strategies = false;             // ATZ_F_STRATEGIES: also try zlib's other strategies (changes the ATZ file vs the reference)
    bool smallWindows = false;           // ATZ_SCAN_SMALL_WINDOWS: also accept CINFO 0 and 1 headers (the reference can still reconstruct)
    bool png = false;                    // ATZ_SCAN_PNG_IDAT: also find zlib streams split over PNG IDAT chunks (changes the ATZ file vs the reference)
    bool apng = false;                   // ATZ_SCAN_APNG_FDAT: also find zlib streams split over APNG fdAT chunks (changes the ATZ file vs the reference)
    int nested = 0;                      // ATZ_F_NESTED_DEPTH: also recompress zlib streams inside recompressed ones, this many levels deep (changes the ATZ file vs the reference)
};

struct zlibParamPack {
    zlibParamPack() {}
    zlibParamPack(uint8_t c, uint8_t w, uint8_t m) : clevel(c), window(w), memlevel(m) {}
    uint8_t clevel = 9, window = 15, memlevel = 9;
};

class streamOffset {
  public:
    streamOffset() = delete;
    streamOffset(uint64_t os, int ot, uint64_t sl, uint64_t il)
        : zlibparams(9, 15, 9), offset(os), offsetType(ot), streamLength(sl), inflatedLength(il), identBytes(0), firstDiffByte(-1),
          recomp(false), atzInfos(0) {}
    zlibParamPack zlibparams;
    uint64_t offset;
    int offsetType;
    uint64_t streamLength;
    uint64_t inflatedLength;
    uint64_t identBytes;
    int_fast64_t firstDiffByte;            // first mismatching byte, relative to the stream start; -1 = none
    std::vector<uint64_t> diffByteOffsets; // delta-encoded positions (first entry 0)
    std::vector<uint8_t> diffByteVal;      // the original bytes at those positions
    bool recomp;
    uint64_t atzInfos;                     // reconstruct: offset of the inflated payload inside the ATZ file
    // antiz_b200 extension (ATZ_SCAN_PNG_IDAT, ATZ_SCAN_APNG_FDAT): a stream split over PNG IDAT or APNG fdAT chunks has npieces >= 2
    // pieces in the file, `frame` bytes of chunk framing between two (12: IDAT, 16: fdAT); streamLength is the sum of the pieces
    std::vector<uint32_t> pieces;
    uint32_t frame = 12;
    uint64_t gapsAt = 0;                   // reconstruct: offset of the framing bytes inside the ATZ file
    uint64_t spanLength() const { return streamLength + (pieces.empty() ? 0 : (uint64_t)frame * (pieces.size() - 1)); }   // bytes of the original the stream covers
};

class fileOffset {   // unused by the reference's live code; kept for source compatibility
  public:
    fileOffset() = delete;
    fileOffset(uint64_t os, int ot) : offset(os), offsetType(ot) {}
    uint64_t offset;
    int offsetType;
};

} // namespace ATZdata
#endif

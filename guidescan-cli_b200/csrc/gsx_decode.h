// gsx_decode.h -- the device half of gsx_decode_database (gsx_decode.cu): a SAM complete database's of:H: lists back into
// off-target rows.  The host half (record splitting, checks, text) is in gsx_format.cpp.
#ifndef GSX_DECODE_H
#define GSX_DECODE_H
#include "gsx_types.h"
#include <cstdint>
#include <memory>
#include <string>
#include <vector>

namespace gsx {

// one decoded record's guide: protospacer + PAM column in guide orientation (SEQ with FLAG 16 undone)
struct DecodeGuide {
    char seq[kMaxQ + kMaxPamLen];
    uint8_t qlen, plen;
    uint8_t pad[6];
};

// the PAMs a listed site may carry besides the record's own PAM column (-a), all of the column's length; N matches anything
struct DecodePams {
    uint32_t n;
    char p[kMaxPams][kMaxPamLen];
};

// first failure of a batch (lowest entry): what, and at which 16-digit entry of the batch
enum : uint32_t { kDecodeBadHex = 1, kDecodeBadGroup = 2, kDecodeOutside = 3, kDecodeDistance = 4, kDecodePam = 5 };

// One batch: `text` holds the SAM bytes of its records; record r's of:H: value starts at byte rec_hex[r] and holds entries
// [rec_entry[r], rec_entry[r + 1]) of the batch (16 hex digits each).
struct DecodeBatchIn {
    const char* text; size_t text_bytes;
    const uint64_t* rec_hex; const uint32_t* rec_entry; const DecodeGuide* guides; uint32_t n_rec;
};

// grow-only pinned host memory
struct PinnedBuf {
    void* p = nullptr; size_t cap = 0;
    PinnedBuf() = default;
    PinnedBuf(const PinnedBuf&) = delete; PinnedBuf& operator=(const PinnedBuf&) = delete;
    void* need(size_t bytes);         // throws gsx::SiteError
    ~PinnedBuf();
};

// Rows of a batch in host memory (pinned, owned by this object and reused by the next run into it): rows of record r are
// [rec_row[r], rec_row[r + 1]), in list order; match has `stride` bytes per row.
struct DecodeRows {
    uint32_t n_rows = 0, stride = 0;
    const uint32_t* rec_row = nullptr;
    const int32_t* chr = nullptr; const uint32_t* pos1 = nullptr; const uint8_t* strand = nullptr; const uint8_t* distance = nullptr;
    const float* cfd = nullptr; const char* match = nullptr;
    // err_code 0: every entry decoded; else the batch's first failure (a digit that is not hex before any other): its entry, the
    // entry's value, and for kDecodeDistance the listed distance and the mismatches found
    uint32_t err_code = 0, err_entry = 0, err_listed = 0, err_found = 0; int64_t err_value = 0;
    double ms = 0;                                                    // device events: first upload to last copy
    PinnedBuf buf[7];
};

// The genome (one byte per base, the index builder's upper-case text) and the chromosome table live on `device` for the object's
// lifetime; run() takes the device's turn (gsx_host.h device_turn) from its first copy to its last.  Throws gsx::SiteError.
class DecodeDevice {
public:
    DecodeDevice(int device, const uint8_t* genome, uint64_t genome_length, const std::vector<Chrom>& chroms, const DecodePams& pams);
    ~DecodeDevice();
    void run(const DecodeBatchIn& in, DecodeRows& out);
private:
    struct Impl; std::unique_ptr<Impl> d_;
};

}  // namespace gsx
#endif

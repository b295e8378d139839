// gsx_decode.cu -- the device half of gsx_decode_database: the of:H: lists of a SAM complete database (format_sam_guide in
// gsx_format.cpp: per distance d = 0, 1, ..., m the group [abs positions...] [d] [-(G+1)], 16 little-endian hex digits per value)
// back into off-target rows.  Per batch:
//   decode_hex_kernel    one thread per 16-digit entry: hex -> int64, delimiter flag
//   (exclusive scan of the flags: delimiters before each entry = its group inside the record, and its row: entry - 2 * delimiters)
//   decode_sites_kernel  one thread per entry: checks the group structure; for a position, resolve_abs, the site's window from the
//                        concatenated genome, the match string in guide orientation, mismatches and PAM against the list, CFD
// The coordinate and CFD arithmetic is gsx_core.h's, the same calls score_hit makes.
#include "../../include/gsx.h"
#include "gsx_core.h"
#include "gsx_decode.h"
#include "gsx_iupac.h"
#include "gsx_host.h"
#include "gsx_sites.h"
#include "cfd_tables.h"
#include <cub/cub.cuh>
#include <cuda_runtime.h>
#include <string>

namespace gsx {

// the search path's CFD tables (gsx_kernels.cu keeps its own copy in that translation unit; both come from cfd_tables.h)
__constant__ double c_dec_cfd_mm[4 * 4 * 20];
__constant__ double c_dec_cfd_pam[4 * 4];

namespace {

struct DecodeArgs {
    const unsigned char* genome; uint64_t G;
    const Chrom* chroms; uint32_t n_chr;
    const uint32_t* rec_entry; const DecodeGuide* guides; uint32_t n_rec, n_entries;
    const int64_t* val; const uint32_t* is_delim; const uint32_t* before;
    DecodePams pams;
    uint32_t stride;
    uint32_t* rec_row; int32_t* chr; uint32_t* pos1; uint8_t* strand; uint8_t* distance; float* cfd; char* match;
    unsigned long long* err;
};

__device__ __forceinline__ uint32_t record_of(const uint32_t* rec_entry, uint32_t n_rec, uint32_t e) {   // last r with rec_entry[r] <= e
    uint32_t lo = 0, hi = n_rec;
    while (hi - lo > 1) { const uint32_t mid = (lo + hi) >> 1; if (rec_entry[mid] <= e) lo = mid; else hi = mid; }
    return lo;
}
__device__ __forceinline__ int hex_digit(unsigned char c) {
    const unsigned char l = c | 32u;
    return c >= '0' && c <= '9' ? c - '0' : (l >= 'a' && l <= 'f' ? l - 'a' + 10 : -1);
}
// the batch's first failure: entry << 24 | listed distance << 16 | mismatches found << 8 | code (the distances for kDecodeDistance)
__device__ __forceinline__ void fail(unsigned long long* err, uint32_t e, uint32_t code, uint32_t listed = 0, uint32_t found = 0) {
    atomicMin(err, ((unsigned long long)e << 24) | ((listed & 0xffu) << 16) | ((found & 0xffu) << 8) | code);
}

__global__ void decode_hex_kernel(const unsigned char* __restrict__ text, const uint64_t* __restrict__ rec_hex, const uint32_t* __restrict__ rec_entry,
                                  uint32_t n_rec, uint32_t n_entries, int64_t delim, int64_t* __restrict__ val, uint32_t* __restrict__ is_delim,
                                  unsigned long long* err_hex) {
    for (uint32_t e = blockIdx.x * blockDim.x + threadIdx.x; e < n_entries; e += gridDim.x * blockDim.x) {
        const uint32_t r = record_of(rec_entry, n_rec, e);
        const unsigned char* p = text + rec_hex[r] + 16ull * (e - rec_entry[r]);
        uint64_t v = 0; int bad = 0;
        for (int b = 0; b < 8; b++) {                                         // byte b = digits 2b (high nibble), 2b + 1
            const int h = hex_digit(p[2 * b]), l = hex_digit(p[2 * b + 1]);
            bad |= h | l;
            v |= (uint64_t)(((h << 4) | l) & 0xff) << (8 * b);
        }
        if (bad < 0) fail(err_hex, e, kDecodeBadHex);
        val[e] = (int64_t)v;
        is_delim[e] = bad >= 0 && (int64_t)v == delim;
    }
}

// N accepts any site character, a class letter (R, Y, ..., V) its member bases, any other letter itself (gsx_iupac.h)
__device__ __forceinline__ bool pam_fits(const char* pam, const char* site, uint32_t plen) {
    for (uint32_t i = 0; i < plen; i++) if (!iupac_pam_fits(pam[i], site[i])) return false;
    return true;
}

__device__ void decode_entry(const DecodeArgs& a, uint32_t e) {
    const uint32_t r = record_of(a.rec_entry, a.n_rec, e);
    const uint32_t e0 = a.rec_entry[r], e1 = a.rec_entry[r + 1];
    const uint32_t before = a.before[e], dl = a.is_delim[e];
    if (e == e0) a.rec_row[r] = e - 2 * before;
    if (e + 1 == a.n_entries) a.rec_row[a.n_rec] = e + 1 - 2 * (before + dl);
    if (dl) { if (e == e0 || a.is_delim[e - 1]) fail(a.err, e, kDecodeBadGroup); return; }      // a group needs its distance
    if (e + 1 == e1) { fail(a.err, e, kDecodeBadGroup); return; }                                  // the list ends with a delimiter
    const uint32_t t = before - a.before[e0];                                                      // group = listed distance
    if (a.is_delim[e + 1]) { if (a.val[e] != (int64_t)t) fail(a.err, e, kDecodeBadGroup); return; }   // the group's distance
    // a position of group t
    const uint32_t row = e - 2 * before;
    const DecodeGuide g = a.guides[r];
    const uint32_t q = g.qlen, L = q + g.plen;
    const int64_t abs = a.val[e];
    uint64_t s;
    const bool fwd = abs >= 0;
    if (fwd) { if ((uint64_t)abs >= a.G || (uint64_t)abs + 1 < L) { fail(a.err, e, kDecodeOutside); return; } s = (uint64_t)abs + 1 - L; }
    else { if (abs < -(int64_t)a.G || (uint64_t)(-abs) + L > a.G) { fail(a.err, e, kDecodeOutside); return; } s = (uint64_t)(-abs); }
    uint32_t pos1 = 0; uint8_t sc = '+';
    const int chr = resolve_abs(a.chroms, a.n_chr, abs, q, g.plen, &pos1, &sc);
    if (chr < 0) { fail(a.err, e, kDecodeOutside); return; }
    char m[kMaxQ + kMaxPamLen];
    uint32_t mm = 0;
    for (uint32_t i = 0; i < L; i++) {                                        // the site in guide orientation
        char c = fwd ? (char)a.genome[s + i] : complement_char((char)a.genome[s + L - 1 - i]);
        if (i < q && c != g.seq[i]) { mm++; if (c >= 'A' && c <= 'Z') c = (char)(c + 32); }
        m[i] = c;
    }
    if (mm != t) { fail(a.err, e, kDecodeDistance, t, mm); return; }
    bool pam_ok = pam_fits(g.seq + q, m + q, g.plen);
    for (uint32_t k = 0; k < a.pams.n && !pam_ok; k++) pam_ok = pam_fits(a.pams.p[k], m + q, g.plen);
    if (!pam_ok) { fail(a.err, e, kDecodePam); return; }
    a.chr[row] = chr; a.pos1[row] = pos1; a.strand[row] = sc; a.distance[row] = (uint8_t)t;
    a.cfd[row] = cfd_score(g.seq, q, m, L, c_dec_cfd_mm, c_dec_cfd_pam);
    char* out = a.match + (size_t)row * a.stride;
    for (uint32_t i = 0; i < L; i++) out[i] = m[i];
}

__global__ void decode_sites_kernel(const DecodeArgs a) {
    for (uint32_t e = blockIdx.x * blockDim.x + threadIdx.x; e < a.n_entries; e += gridDim.x * blockDim.x) decode_entry(a, e);
}

#define DCK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) throw SiteError{GSX_ERR_CUDA, std::string(#x ": ") + cudaGetErrorString(e_)}; } while (0)

// grow-only device / pinned host buffers
struct DevBuf {
    void* p = nullptr; size_t cap = 0;
    void* need(size_t bytes) {
        if (bytes > cap) { cudaFree(p); p = nullptr; cap = bytes + bytes / 4 + 256; DCK(cudaMalloc(&p, cap)); }
        return p;
    }
    ~DevBuf() { cudaFree(p); }
};
}  // namespace

void* PinnedBuf::need(size_t bytes) {
    if (bytes > cap) { cudaFreeHost(p); p = nullptr; cap = bytes + bytes / 4 + 256; DCK(cudaHostAlloc(&p, cap, cudaHostAllocDefault)); }
    return p;
}
PinnedBuf::~PinnedBuf() { cudaFreeHost(p); }

struct DecodeDevice::Impl {
    int device = 0; uint64_t G = 0; uint32_t n_chr = 0; DecodePams pams{};
    DevBuf genome, chroms, text, rec_hex, rec_entry, guides, val, is_delim, before, scan_tmp, rec_row, chr, pos1, strand, distance, cfd, match, err;
    cudaStream_t stream = nullptr; cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    ~Impl() {
        cudaSetDevice(device);
        if (ev0) cudaEventDestroy(ev0);
        if (ev1) cudaEventDestroy(ev1);
        if (stream) cudaStreamDestroy(stream);
    }
};

DecodeDevice::DecodeDevice(int device, const uint8_t* genome, uint64_t G, const std::vector<Chrom>& chroms, const DecodePams& pams) : d_(new Impl()) {
    Impl& D = *d_;
    D.device = device; D.G = G; D.n_chr = (uint32_t)chroms.size(); D.pams = pams;
    DCK(cudaSetDevice(device));
    DCK(cudaStreamCreateWithFlags(&D.stream, cudaStreamNonBlocking));
    DCK(cudaEventCreate(&D.ev0)); DCK(cudaEventCreate(&D.ev1));
    DCK(cudaMemcpyToSymbol(c_dec_cfd_mm, GSX_CFD_MM, sizeof(c_dec_cfd_mm)));
    DCK(cudaMemcpyToSymbol(c_dec_cfd_pam, GSX_CFD_PAM, sizeof(c_dec_cfd_pam)));
    std::unique_lock<std::mutex> turn = device_turn(device);
    DCK(cudaMemcpyAsync(D.genome.need(G), genome, G, cudaMemcpyHostToDevice, D.stream));
    DCK(cudaMemcpyAsync(D.chroms.need(chroms.size() * sizeof(Chrom)), chroms.data(), chroms.size() * sizeof(Chrom), cudaMemcpyHostToDevice, D.stream));
    DCK(cudaStreamSynchronize(D.stream));
}
DecodeDevice::~DecodeDevice() { if (d_) cudaSetDevice(d_->device); }

void DecodeDevice::run(const DecodeBatchIn& in, DecodeRows& out) {
    Impl& D = *d_;
    const uint32_t E = in.n_rec ? in.rec_entry[in.n_rec] : 0;
    out.n_rows = 0; out.rec_row = nullptr; out.chr = nullptr; out.pos1 = nullptr; out.strand = nullptr; out.distance = nullptr;
    out.cfd = nullptr; out.match = nullptr; out.err_code = 0; out.err_listed = 0; out.err_found = 0; out.err_entry = 0; out.err_value = 0; out.ms = 0;
    uint32_t stride = 1;
    for (uint32_t r = 0; r < in.n_rec; r++) stride = std::max<uint32_t>(stride, (uint32_t)in.guides[r].qlen + in.guides[r].plen);
    out.stride = stride;
    if (!E) { static const uint32_t zero[1] = {0}; out.rec_row = zero; return; }
    DCK(cudaSetDevice(D.device));
    cudaStream_t s = D.stream;
    // sizes first (allocation outside the device's turn)
    char* d_text = (char*)D.text.need(in.text_bytes);
    uint64_t* d_rec_hex = (uint64_t*)D.rec_hex.need(in.n_rec * sizeof(uint64_t));
    uint32_t* d_rec_entry = (uint32_t*)D.rec_entry.need((in.n_rec + 1) * sizeof(uint32_t));
    DecodeGuide* d_guides = (DecodeGuide*)D.guides.need(in.n_rec * sizeof(DecodeGuide));
    int64_t* d_val = (int64_t*)D.val.need((size_t)E * 8);
    uint32_t* d_is_delim = (uint32_t*)D.is_delim.need((size_t)E * 4);
    uint32_t* d_before = (uint32_t*)D.before.need((size_t)E * 4);
    size_t scan_bytes = 0;
    DCK(cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, d_is_delim, d_before, (int)E, s));
    void* d_scan = D.scan_tmp.need(scan_bytes);
    DecodeArgs a{};
    a.genome = (const unsigned char*)D.genome.p; a.G = D.G; a.chroms = (const Chrom*)D.chroms.p; a.n_chr = D.n_chr;
    a.rec_entry = d_rec_entry; a.guides = d_guides; a.n_rec = in.n_rec; a.n_entries = E;
    a.val = d_val; a.is_delim = d_is_delim; a.before = d_before; a.pams = D.pams; a.stride = stride;
    a.rec_row = (uint32_t*)D.rec_row.need((in.n_rec + 1) * sizeof(uint32_t));
    a.chr = (int32_t*)D.chr.need((size_t)E * 4); a.pos1 = (uint32_t*)D.pos1.need((size_t)E * 4);
    a.strand = (uint8_t*)D.strand.need(E); a.distance = (uint8_t*)D.distance.need(E);
    a.cfd = (float*)D.cfd.need((size_t)E * 4); a.match = (char*)D.match.need((size_t)E * stride);
    a.err = (unsigned long long*)D.err.need(16);
    unsigned long long* d_err_hex = a.err + 1;                               // (bad digits first: a broken delimiter misleads the group checks)
    // the rows' pinned buffers for as many rows as entries, before the turn (cudaHostAlloc costs about half a second per GiB)
    uint32_t* h_rec_row = (uint32_t*)out.buf[0].need((in.n_rec + 1) * sizeof(uint32_t));
    int32_t* h_chr = (int32_t*)out.buf[1].need((size_t)E * 4); uint32_t* h_pos1 = (uint32_t*)out.buf[2].need((size_t)E * 4);
    uint8_t* h_strand = (uint8_t*)out.buf[3].need(E); uint8_t* h_distance = (uint8_t*)out.buf[4].need(E);
    float* h_cfd = (float*)out.buf[5].need((size_t)E * 4); char* h_match = (char*)out.buf[6].need((size_t)E * stride);
    unsigned long long h_err[2] = {~0ull, ~0ull};
    const int64_t delim = -(int64_t)(D.G + 1);
    const int blocks = (int)std::min<uint64_t>((E + 255) / 256, 148ull * 16);

    std::unique_lock<std::mutex> turn = device_turn(D.device);
    DCK(cudaEventRecord(D.ev0, s));
    DCK(cudaMemcpyAsync(d_text, in.text, in.text_bytes, cudaMemcpyHostToDevice, s));
    DCK(cudaMemcpyAsync(d_rec_hex, in.rec_hex, in.n_rec * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
    DCK(cudaMemcpyAsync(d_rec_entry, in.rec_entry, (in.n_rec + 1) * sizeof(uint32_t), cudaMemcpyHostToDevice, s));
    DCK(cudaMemcpyAsync(d_guides, in.guides, in.n_rec * sizeof(DecodeGuide), cudaMemcpyHostToDevice, s));
    DCK(cudaMemcpyAsync(a.err, h_err, 16, cudaMemcpyHostToDevice, s));
    decode_hex_kernel<<<blocks, 256, 0, s>>>((const unsigned char*)d_text, d_rec_hex, d_rec_entry, in.n_rec, E, delim, d_val, d_is_delim, d_err_hex);
    DCK(cudaGetLastError());
    DCK(cub::DeviceScan::ExclusiveSum(d_scan, scan_bytes, d_is_delim, d_before, (int)E, s));
    decode_sites_kernel<<<blocks, 256, 0, s>>>(a);
    DCK(cudaGetLastError());
    DCK(cudaMemcpyAsync(h_err, a.err, 16, cudaMemcpyDeviceToHost, s));
    DCK(cudaMemcpyAsync(h_rec_row, a.rec_row, (in.n_rec + 1) * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
    DCK(cudaStreamSynchronize(s));
    out.rec_row = h_rec_row;
    const unsigned long long fe = h_err[1] != ~0ull ? h_err[1] : h_err[0];
    if (fe != ~0ull) {
        out.err_code = (uint32_t)(fe & 0xff); out.err_found = (uint32_t)((fe >> 8) & 0xff); out.err_listed = (uint32_t)((fe >> 16) & 0xff);
        out.err_entry = (uint32_t)(fe >> 24);
        DCK(cudaMemcpyAsync(&out.err_value, d_val + out.err_entry, 8, cudaMemcpyDeviceToHost, s));
        DCK(cudaStreamSynchronize(s));
        return;
    }
    const uint32_t n = h_rec_row[in.n_rec];
    out.n_rows = n;
    if (n) {
        DCK(cudaMemcpyAsync(h_chr, a.chr, (size_t)n * 4, cudaMemcpyDeviceToHost, s));
        DCK(cudaMemcpyAsync(h_pos1, a.pos1, (size_t)n * 4, cudaMemcpyDeviceToHost, s));
        DCK(cudaMemcpyAsync(h_strand, a.strand, n, cudaMemcpyDeviceToHost, s));
        DCK(cudaMemcpyAsync(h_distance, a.distance, n, cudaMemcpyDeviceToHost, s));
        DCK(cudaMemcpyAsync(h_cfd, a.cfd, (size_t)n * 4, cudaMemcpyDeviceToHost, s));
        DCK(cudaMemcpyAsync(h_match, a.match, (size_t)n * stride, cudaMemcpyDeviceToHost, s));
    }
    DCK(cudaEventRecord(D.ev1, s));
    DCK(cudaStreamSynchronize(s));
    if (turn.owns_lock()) turn.unlock();                                     // (GSX_DEVICE_LOCK=0: no turn is held)
    float ms = 0; cudaEventElapsedTime(&ms, D.ev0, D.ev1); out.ms = ms;
    out.chr = h_chr; out.pos1 = h_pos1; out.strand = h_strand; out.distance = h_distance; out.cfd = h_cfd; out.match = h_match;
}

}  // namespace gsx

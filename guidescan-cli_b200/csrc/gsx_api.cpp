// gsx_api.cpp -- C ABI (include/gsx.h): index upload, batched enumerate on 1..N devices, result arenas.
// Host orchestration only; all arithmetic of the path runs in the kernels of gsx_kernels.cu.  No CPU fallback.
#include "../../include/gsx.h"
#include "gsx_host.h"
#include "gsx_core.h"
#include "gsx_iupac.h"
#include <cuda_runtime.h>
#include <algorithm>
#include <chrono>
#include <climits>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <stdexcept>
#include <string>
#include <thread>
#include <type_traits>
#include <sys/stat.h>
#include <vector>

using namespace gsx;

static thread_local std::string g_err;
static int fail(int code, const std::string& msg) { g_err = msg; return code; }
int gsx_set_error(int code, const std::string& msg) { return fail(code, msg); }      // for the other translation units

struct CudaError : std::runtime_error { using std::runtime_error::runtime_error; };
#define CK(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) throw CudaError(std::string(#call) + ": " + cudaGetErrorString(e__)); } while (0)

static int env_int(const char* name, int dflt) { const char* v = getenv(name); return v && *v ? atoi(v) : dflt; }

// One call's guide packing and host-side result assembly run under the next call's kernels, and two sweeps never share -- and
// thrash -- the L2-resident slices; the PAM scan of gsx_enumerate_genome takes the same turn for its chromosome upload.
// GSX_DEVICE_LOCK=0 turns it off.
std::unique_lock<std::mutex> gsx::device_turn(int device) {
    static std::mutex device_mu[64];
    if (!env_int("GSX_DEVICE_LOCK", 1)) return std::unique_lock<std::mutex>();
    return std::unique_lock<std::mutex>(device_mu[device & 63]);
}

extern "C" const char* gsx_last_error(void) { return g_err.c_str(); }
extern "C" const char* gsx_version(void) { return "2.0.0"; }
extern "C" void gsx_free(void* p) { free(p); }
extern "C" int gsx_device_count(void) { int n = 0; if (cudaGetDeviceCount(&n) != cudaSuccess) return 0; return n; }

extern "C" void gsx_params_default(gsx_params* p) {
    memset(p, 0, sizeof *p);
    p->mismatches = 3; p->max_bulge_size = 1; p->threshold = -1; p->max_off_targets = -1;
}

// ---------------------------------------------------------------------------------------------------------
// index
// ---------------------------------------------------------------------------------------------------------
template <class T> static void* upload(const std::vector<T>& v, size_t& n_bytes, uint64_t& total) {
    void* d = nullptr; size_t n = std::max<size_t>(v.size(), 1) * sizeof(T);
    CK(cudaMalloc(&d, n));
    if (!v.empty()) CK(cudaMemcpy(d, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
    else CK(cudaMemset(d, 0, n));                                            // (an empty table still has one, defined, element)
    n_bytes = n; total += n;
    return d;
}

static double seconds_since(std::chrono::steady_clock::time_point t0) { return std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count(); }

// device pointers of a strand -> the view the kernels take
static void bind_strand(DeviceStrand& d) {
    d.d.blocks = (const OccBlock*)d.blocks; d.d.sa_samples = (const uint32_t*)d.sa;
    d.d.exc_rows = (const uint32_t*)d.exc_rows; d.d.exc_lf = (const uint32_t*)d.exc_lf; d.d.n_rows = (const uint32_t*)d.n_rows;
    d.d.lines = (const unsigned char*)d.lines; d.d.sum0 = (const unsigned char*)d.sum0; d.d.sum1 = (const unsigned char*)d.sum1;
    d.d.sum2 = (const unsigned char*)d.sum2; d.d.ftab = d.ftab;
}

// The whole index on ONE device: the host arrays go up, everything else (jump table, look-ahead lines, pattern summaries: 64 of
// the 69 GB of a 3.1 Gb genome) is derived there by kernels.
static void build_device_index(gsx_index* ix, DeviceIndex& di) {
    CK(cudaSetDevice(di.device));
    cudaDeviceProp prop; CK(cudaGetDeviceProperties(&prop, di.device));
    di.sm_count = prop.multiProcessorCount;
    CK(upload_cfd_tables());
    for (int s = 0; s < 2; s++) {
        const HostStrand& h = ix->host.st[s];
        DeviceStrand& d = di.st[s];
        d.blocks = upload(h.blocks, d.blocks_bytes, di.bytes); d.sa = upload(h.sa_samples, d.sa_bytes, di.bytes);
        d.exc_rows = upload(h.exc_rows, d.exc_rows_bytes, di.bytes); d.exc_lf = upload(h.exc_lf, d.exc_lf_bytes, di.bytes);
        d.n_rows = upload(h.n_rows, d.n_rows_bytes, di.bytes);
        d.exc_map = upload(build_exc_map(h), d.exc_map_bytes, di.bytes);
        bind_strand(d);
        d.d.n = (uint32_t)h.n; d.d.n_exc = (uint32_t)h.exc_rows.size(); d.d.n_nrows = (uint32_t)h.n_rows.size();
        d.d.sa_shift = h.sa_shift;
        for (int c = 0; c < 5; c++) d.d.C[c] = h.C[c];
        d.d.exc_lo = h.exc_rows.empty() ? 0xFFFFFFFFu : h.exc_rows.front();
        d.d.exc_hi = h.exc_rows.empty() ? 0u : h.exc_rows.back();
        d.d.blk_shift = 5; d.d.ftab_L = 0;
        {
            // k-mer jump table: depth L such that a level-L interval still holds a handful of rows
            int L = env_int("GSX_FTAB", -1);
            if (L < 0) { L = 0; uint64_t v = h.n; while (v >= 4) { v >>= 2; L++; } L -= 1; if (L > 14) L = 14; if (L < 6) L = 0; }
            if (L > 16) L = 16;
            if (L >= 4) {
                void* tmp = nullptr;
                d.ftab_bytes = (size_t)8 << (2 * L);
                CK(cudaMalloc(&d.ftab, d.ftab_bytes));
                CK(cudaMalloc(&tmp, d.ftab_bytes));
                CK(launch_build_ftab(d.d, (uint32_t)L, d.ftab, tmp, 0));
                CK(cudaDeviceSynchronize());
                cudaFree(tmp);
                d.d.ftab = d.ftab; d.d.ftab_L = (uint32_t)L; di.bytes += d.ftab_bytes;
            }
        }
        if (env_int("GSX_LOOKAHEAD", 1)) {
            // second copy for narrow intervals: one 128-byte line per 64 rows = OccBlock + look-ahead planes t1..t6,
            // derived on the device by LF walks over the packed blocks (t7, t8 into a scratch array for the summaries)
            const uint32_t nb = (uint32_t)h.blocks.size();
            const bool summaries = d.d.ftab && env_int("GSX_SWEEP_SUMMARY", 1);
            void* tail = nullptr;
            d.lines_bytes = (size_t)nb * 128;
            CK(cudaMalloc(&d.lines, d.lines_bytes));
            if (summaries && env_int("GSX_SWEEP_TAIL", 1)) CK(cudaMalloc(&tail, (size_t)nb * 32));
            CK(launch_build_lookahead(d.d, (unsigned char*)d.lines, (unsigned char*)tail, nb, 0));
            CK(cudaDeviceSynchronize());
            d.d.lines = (const unsigned char*)d.lines; di.bytes += d.lines_bytes;
            if (summaries) {
                // pattern summaries for the slice-major front end (sweep_kernel): 2 x 32 (+ 16) bytes per jump-table entry
                const uint64_t n_entries = 1ull << (2 * d.d.ftab_L);
                d.sum0_bytes = d.sum1_bytes = n_entries * 32;
                CK(cudaMalloc(&d.sum0, d.sum0_bytes)); CK(cudaMalloc(&d.sum1, d.sum1_bytes));
                if (tail) { d.sum2_bytes = n_entries * 16; CK(cudaMalloc(&d.sum2, d.sum2_bytes)); }
                CK(launch_build_summary(d.ftab, (const unsigned char*)d.lines, (const unsigned char*)tail, (unsigned char*)d.sum0,
                                        (unsigned char*)d.sum1, (unsigned char*)d.sum2, n_entries, 0));
                CK(cudaDeviceSynchronize());
                di.bytes += n_entries * (tail ? 80 : 64);
            }
            cudaFree(tail);
        }
        bind_strand(d);
    }
    size_t cb = 0;
    di.chroms = (Chrom*)upload(ix->chroms, cb, di.bytes);
}

// A further device receives the finished arrays of the first one by peer copies (NVLink / NVSwitch: 69 GB in well under a
// second per device; staged through the host by the driver where peer access is not available) instead of deriving them
// again -- 64 of the 69 GB of a 3.1 Gb index are derived data and took ~35 s per device.
static void replicate_device_index(const gsx_index* ix, const DeviceIndex& src, DeviceIndex& dst, cudaStream_t stream) {
    CK(cudaSetDevice(dst.device));
    cudaDeviceProp prop; CK(cudaGetDeviceProperties(&prop, dst.device));
    dst.sm_count = prop.multiProcessorCount;
    CK(upload_cfd_tables());
    int can = 0;
    if (cudaDeviceCanAccessPeer(&can, dst.device, src.device) == cudaSuccess && can) {
        cudaError_t e = cudaDeviceEnablePeerAccess(src.device, 0);
        if (e != cudaSuccess) cudaGetLastError();                            // (already enabled / not supported: the copy still works)
    }
    for (int s = 0; s < 2; s++) {
        const DeviceStrand& a = src.st[s]; DeviceStrand& d = dst.st[s];
        d.d = a.d;
#define GSX_COPY(name) if (a.name) { d.name##_bytes = a.name##_bytes; CK(cudaMalloc(&d.name, d.name##_bytes)); \
                                     CK(cudaMemcpyPeerAsync(d.name, dst.device, a.name, src.device, d.name##_bytes, stream)); dst.bytes += d.name##_bytes; }
        GSX_STRAND_ARRAYS(GSX_COPY)
#undef GSX_COPY
        bind_strand(d);
    }
    const size_t cb = std::max<size_t>(ix->chroms.size(), 1) * sizeof(Chrom);
    CK(cudaMalloc(&dst.chroms, cb));
    CK(cudaMemcpyPeerAsync(dst.chroms, dst.device, src.chroms, src.device, cb, stream)); dst.bytes += cb;
}

static void upload_index(gsx_index* ix, const int* devices, int n_devices) {
    ix->chroms.clear();
    uint64_t start = 0;
    for (size_t i = 0; i < ix->host.chr_lens.size(); i++) { ix->chroms.push_back({start, ix->host.chr_lens[i]}); start += ix->host.chr_lens[i]; }
    std::vector<int> devs;
    if (!devices || n_devices <= 0) devs.push_back(0); else devs.assign(devices, devices + n_devices);
    ix->dev.clear(); ix->dev.reserve(devs.size());
    auto t0 = std::chrono::steady_clock::now();
    {
        DeviceIndex di; di.device = devs[0];
        ix->dev.push_back(di);                                               // (in the list first: a failure below frees what was allocated)
        build_device_index(ix, ix->dev[0]);
    }
    ix->open_seconds[1] = seconds_since(t0);
    t0 = std::chrono::steady_clock::now();
    std::vector<cudaStream_t> streams;
    struct Cleanup { std::vector<cudaStream_t>& s; ~Cleanup() { for (auto x : s) cudaStreamDestroy(x); } } cleanup{streams};
    for (size_t k = 1; k < devs.size(); k++) {
        DeviceIndex di; di.device = devs[k];
        for (size_t j = 0; j < k; j++) if (ix->dev[j].device == devs[k] && ix->dev[j].alias_of < 0) { di.alias_of = (int)j; break; }
        ix->dev.push_back(di);
        DeviceIndex& d = ix->dev.back();
        if (d.alias_of >= 0) {                                               // the same device named twice: two job slots over one copy
            const DeviceIndex& a = ix->dev[d.alias_of];
            d.sm_count = a.sm_count; d.st[0] = a.st[0]; d.st[1] = a.st[1]; d.chroms = a.chroms; d.bytes = a.bytes;
            continue;
        }
        CK(cudaSetDevice(d.device));
        cudaStream_t st; CK(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking)); streams.push_back(st);
        replicate_device_index(ix, ix->dev[0], d, st);                       // (asynchronous: all replicas are filled concurrently)
    }
    for (auto st : streams) CK(cudaStreamSynchronize(st));
    ix->open_seconds[2] = seconds_since(t0);
}

static void free_device_index(DeviceIndex& di) {
    if (di.alias_of >= 0) return;
    cudaSetDevice(di.device);
    cudaDeviceSynchronize();                                                 // (peer copies of a failed open may still be in flight)
    for (int s = 0; s < 2; s++) {
#define GSX_FREE(name) cudaFree(di.st[s].name); di.st[s].name = nullptr;
        GSX_STRAND_ARRAYS(GSX_FREE)
#undef GSX_FREE
    }
    cudaFree(di.chroms); di.chroms = nullptr;
}

static bool file_exists(const std::string& p) { FILE* f = fopen(p.c_str(), "rb"); if (!f) return false; fclose(f); return true; }
static bool file_newer(const std::string& a, const std::string& b) {      // a modified strictly after b
    struct stat sa, sb;
    if (stat(a.c_str(), &sa) != 0 || stat(b.c_str(), &sb) != 0) return false;
    return sa.st_mtim.tv_sec != sb.st_mtim.tv_sec ? sa.st_mtim.tv_sec > sb.st_mtim.tv_sec : sa.st_mtim.tv_nsec > sb.st_mtim.tv_nsec;
}

static int check_devices(const int* devices, int n_devices) {
    int have = gsx_device_count();
    if (have <= 0) return fail(GSX_ERR_NO_DEVICE, "no CUDA device available (this library has no CPU path)");
    for (int i = 0; devices && i < n_devices; i++)
        if (devices[i] < 0 || devices[i] >= have) return fail(GSX_ERR_ARG, "device ordinal out of range");
    return GSX_OK;
}

// every ABI entry point that can throw runs its body through this: nothing but a status code crosses the boundary
template <class F> static int guarded(F&& body) {
    try { return body(); }
    catch (const CudaError& e) { return fail(GSX_ERR_CUDA, e.what()); }
    catch (const std::bad_alloc&) { return fail(GSX_ERR_NOMEM, "out of host memory"); }
    catch (const std::exception& e) { return fail(GSX_ERR_INTERNAL, e.what()); }
    catch (...) { return fail(GSX_ERR_INTERNAL, "unknown exception"); }
}

static int upload_or_fail(gsx_index* ix, const int* devices, int n_devices, gsx_index** out) {
    const int rc = guarded([&] { upload_index(ix, devices, n_devices); return (int)GSX_OK; });
    if (rc) { const std::string msg = g_err; for (auto& d : ix->dev) free_device_index(d); delete ix; return fail(rc, msg); }
    *out = ix;
    return GSX_OK;
}

extern "C" int gsx_index_open(const char* prefix, const int* devices, int n_devices, gsx_index** out) {
    if (!prefix || !out) return fail(GSX_ERR_ARG, "null argument");
    *out = nullptr;
    std::string p(prefix);
    // both formats at one prefix (`guidescan index --reference-format`): the newer one; <prefix>.gsx needs no conversion
    const bool sdsl = !file_exists(p + ".gsx") || (file_exists(p + ".forward") && file_newer(p + ".forward", p + ".gsx"));
    if (!sdsl || (file_exists(p + ".gs") && file_exists(p + ".forward") && file_exists(p + ".reverse")))
        if (int rc = check_devices(devices, n_devices)) return rc;           // (before reading gigabytes; missing files are reported first, as the reference does)
    gsx_index* ix = new gsx_index();
    const auto t0 = std::chrono::steady_clock::now();
    const int rc = guarded([&] {
        std::string err; bool ok;
        if (sdsl) {
            ok = load_genome_structure(p + ".gs", ix->host, err);
            if (ok && !file_exists(p + ".forward")) { ok = false; err = "No forward index file " + p + ".forward located."; }
            if (ok && !file_exists(p + ".reverse")) { ok = false; err = "No forward index file " + p + ".reverse located."; }   // sic: src/guidescan.cxx:205
            if (ok) {
                std::string e0, e1; bool ok0 = false, ok1 = false;
                auto load = [&](int s, const char* ext, bool& okx, std::string& ex) {
                    try { okx = load_sdsl_strand(p + ext, ix->host.st[s], ex); }
                    catch (const std::exception& e) { okx = false; ex = std::string("malformed index file ") + p + ext + " (" + e.what() + ")"; }
                };
                std::thread t0([&] { load(0, ".forward", ok0, e0); });
                std::thread t1([&] { load(1, ".reverse", ok1, e1); });
                t0.join(); t1.join();
                ok = ok0 && ok1; if (!ok) err = ok0 ? e1 : e0;
            }
        } else ok = load_gsx(p, ix->host, err);
        return ok ? (int)GSX_OK : fail(GSX_ERR_IO, err);
    });
    if (rc) { delete ix; return rc; }
    ix->open_seconds[0] = seconds_since(t0);
    if (int rc2 = check_devices(devices, n_devices)) { delete ix; return rc2; }
    return upload_or_fail(ix, devices, n_devices, out);
}

static int build_from_text(gsx_index* ix, std::vector<uint8_t>& seq, uint32_t sa_shift, const char* save_prefix,
                           const int* devices, int n_devices, gsx_index** out) {
    std::string err;
    if (seq.size() + 1 > 0xFFFFFFFFull) { delete ix; return fail(GSX_ERR_ARG, "genome longer than 2^32 - 2 bases"); }
    if (sa_shift > 12) { delete ix; return fail(GSX_ERR_ARG, "sa_shift must be <= 12"); }
    int dev0 = (devices && n_devices > 0) ? devices[0] : 0;
    const auto t0 = std::chrono::steady_clock::now();
    if (!build_strand_gpu(dev0, seq.data(), seq.size(), sa_shift, ix->host.st[0], err)) { delete ix; return fail(GSX_ERR_CUDA, err); }
    {   // reverse complement of the whole concatenated genome, in place (seq_io.cxx:65-72)
        size_t n = seq.size();
        for (size_t i = 0; i < n / 2; i++) { uint8_t a = seq[i], b = seq[n - 1 - i]; seq[i] = (uint8_t)complement_char((char)b); seq[n - 1 - i] = (uint8_t)complement_char((char)a); }
        if (n & 1) seq[n / 2] = (uint8_t)complement_char((char)seq[n / 2]);
    }
    if (!build_strand_gpu(dev0, seq.data(), seq.size(), sa_shift, ix->host.st[1], err)) { delete ix; return fail(GSX_ERR_CUDA, err); }
    if (save_prefix && !save_gsx(save_prefix, ix->host, err)) { delete ix; return fail(GSX_ERR_IO, err); }
    ix->open_seconds[0] = seconds_since(t0);
    return upload_or_fail(ix, devices, n_devices, out);
}

extern "C" int gsx_index_build(const char* fasta_path, const char* save_prefix, const int* devices, int n_devices, gsx_index** out) {
    if (!fasta_path || !out) return fail(GSX_ERR_ARG, "null argument");
    *out = nullptr;
    if (int rc = check_devices(devices, n_devices)) return rc;
    gsx_index* ix = new gsx_index();
    std::string err; std::vector<uint8_t> seq;
    const int rc = guarded([&] { return read_fasta(fasta_path, seq, ix->host, err) ? (int)GSX_OK : fail(GSX_ERR_IO, err); });
    if (rc) { delete ix; return rc; }
    return guarded([&] { return build_from_text(ix, seq, 6, save_prefix, devices, n_devices, out); });
}

extern "C" int gsx_index_build_text(const uint8_t* text, uint64_t length, const char* const* chr_names, const uint64_t* chr_lengths,
                                    uint32_t n_chr, uint32_t sa_shift, const char* save_prefix, const int* devices, int n_devices,
                                    gsx_index** out) {
    if (!text || !out || !chr_names || !chr_lengths) return fail(GSX_ERR_ARG, "null argument");
    *out = nullptr;
    if (int rc = check_devices(devices, n_devices)) return rc;
    gsx_index* ix = new gsx_index();
    uint64_t tot = 0;
    for (uint32_t i = 0; i < n_chr; i++) { ix->host.chr_names.push_back(chr_names[i]); ix->host.chr_lens.push_back(chr_lengths[i]); tot += chr_lengths[i]; }
    ix->host.genome_length = tot;
    return guarded([&] {
        std::vector<uint8_t> seq(text, text + length);
        return build_from_text(ix, seq, sa_shift, save_prefix, devices, n_devices, out);
    });
}

extern "C" int gsx_index_save_reference_format(const gsx_index* ix, const char* prefix) {
    if (!ix || !prefix) return fail(GSX_ERR_ARG, "null argument");
    return guarded([&] { std::string err; return save_sdsl_index(prefix, ix->host, err) ? (int)GSX_OK : fail(GSX_ERR_IO, err); });
}

extern "C" int gsx_index_close(gsx_index* ix) {
    if (!ix) return GSX_OK;
    for (auto& d : ix->dev) { free_device_index(d); pool_trim(d.device); }
    pool_trim(-1);
    delete ix;
    return GSX_OK;
}
extern "C" uint64_t gsx_index_genome_length(const gsx_index* ix) { return ix->host.genome_length; }
extern "C" uint32_t gsx_index_n_chromosomes(const gsx_index* ix) { return (uint32_t)ix->host.chr_names.size(); }
extern "C" const char* gsx_index_chromosome_name(const gsx_index* ix, uint32_t i) { return ix->host.chr_names[i].c_str(); }
extern "C" uint64_t gsx_index_chromosome_length(const gsx_index* ix, uint32_t i) { return ix->host.chr_lens[i]; }
extern "C" uint64_t gsx_index_device_bytes(const gsx_index* ix) { return ix->dev.empty() ? 0 : ix->dev[0].bytes; }
extern "C" int gsx_index_n_devices(const gsx_index* ix) { return (int)ix->dev.size(); }
extern "C" int gsx_index_open_seconds(const gsx_index* ix, double out[3]) {
    if (!ix || !out) return fail(GSX_ERR_ARG, "null argument");
    for (int i = 0; i < 3; i++) out[i] = ix->open_seconds[i];
    return GSX_OK;
}

extern "C" int gsx_index_device_checksum(const gsx_index* ix, int slot, uint64_t* out) {
    if (!ix || !out || slot < 0 || slot >= (int)ix->dev.size()) return fail(GSX_ERR_ARG, "bad argument");
    return guarded([&] {
        const DeviceIndex& di = ix->dev[slot];
        CK(cudaSetDevice(di.device));
        unsigned long long* d_out = nullptr; CK(cudaMalloc(&d_out, 8)); CK(cudaMemset(d_out, 0, 8));
        unsigned long long seed = 1;
        for (int s = 0; s < 2; s++) {
#define GSX_SUM(name) { seed += 0x100; if (di.st[s].name) CK(launch_checksum(di.st[s].name, di.st[s].name##_bytes, seed, d_out, 0)); }
            GSX_STRAND_ARRAYS(GSX_SUM)
#undef GSX_SUM
        }
        CK(launch_checksum(di.chroms, ix->chroms.size() * sizeof(Chrom), seed + 0x100, d_out, 0));
        unsigned long long h = 0; CK(cudaMemcpy(&h, d_out, 8, cudaMemcpyDeviceToHost)); cudaFree(d_out);
        // the scalars the kernels take by value
        for (int s = 0; s < 2; s++) { const DevStrand& d = di.st[s].d; h += 31ull * d.n + 131ull * d.n_exc + 17ull * d.sa_shift + 7ull * d.ftab_L; for (int c = 0; c < 5; c++) h = h * 1000003ull + d.C[c]; }
        *out = h;
        return (int)GSX_OK;
    });
}

static uint8_t sym_of(char c) { return c == 'A' ? SYM_A : c == 'C' ? SYM_C : c == 'G' ? SYM_G : c == 'T' ? SYM_T : c == 'N' ? SYM_N : SYM_X; }

extern "C" int gsx_index_rank(const gsx_index* ix, int strand, const uint64_t* rows, const char* syms, size_t n, uint64_t* out) {
    if (!ix || ix->dev.empty() || strand < 0 || strand > 1) return fail(GSX_ERR_ARG, "bad argument");
    try {
        const DeviceIndex& di = ix->dev[0];
        CK(cudaSetDevice(di.device));
        std::vector<uint32_t> r(n), o(n); std::vector<uint8_t> s(n);
        for (size_t i = 0; i < n; i++) { if (rows[i] > di.st[strand].d.n) return fail(GSX_ERR_ARG, "row out of range"); r[i] = (uint32_t)rows[i]; s[i] = sym_of(syms[i]); }
        uint32_t *dr, *dout; uint8_t* ds;
        CK(cudaMalloc(&dr, n * 4 + 4)); CK(cudaMalloc(&dout, n * 4 + 4)); CK(cudaMalloc(&ds, n + 4));
        CK(cudaMemcpy(dr, r.data(), n * 4, cudaMemcpyHostToDevice)); CK(cudaMemcpy(ds, s.data(), n, cudaMemcpyHostToDevice));
        CK(launch_rank_query(di.st[strand].d, dr, ds, (uint32_t)n, dout, 0));
        CK(cudaMemcpy(o.data(), dout, n * 4, cudaMemcpyDeviceToHost));
        cudaFree(dr); cudaFree(dout); cudaFree(ds);
        for (size_t i = 0; i < n; i++) out[i] = o[i];
    } catch (const CudaError& e) { return fail(GSX_ERR_CUDA, e.what()); }
    return GSX_OK;
}

extern "C" int gsx_index_locate(const gsx_index* ix, int strand, const uint64_t* rows, size_t n, uint64_t* out) {
    if (!ix || ix->dev.empty() || strand < 0 || strand > 1) return fail(GSX_ERR_ARG, "bad argument");
    try {
        const DeviceIndex& di = ix->dev[0];
        CK(cudaSetDevice(di.device));
        std::vector<uint32_t> r(n), o(n);
        for (size_t i = 0; i < n; i++) { if (rows[i] >= di.st[strand].d.n) return fail(GSX_ERR_ARG, "row out of range"); r[i] = (uint32_t)rows[i]; }
        uint32_t *dr, *dout;
        CK(cudaMalloc(&dr, n * 4 + 4)); CK(cudaMalloc(&dout, n * 4 + 4));
        CK(cudaMemcpy(dr, r.data(), n * 4, cudaMemcpyHostToDevice));
        CK(launch_locate_query(di.st[strand].d, dr, (uint32_t)n, dout, 0));
        CK(cudaMemcpy(o.data(), dout, n * 4, cudaMemcpyDeviceToHost));
        cudaFree(dr); cudaFree(dout);
        for (size_t i = 0; i < n; i++) out[i] = o[i];
    } catch (const CudaError& e) { return fail(GSX_ERR_CUDA, e.what()); }
    return GSX_OK;
}

extern "C" int gsx_index_export_bwt(const gsx_index* ix, int strand, uint8_t* out) {
    if (!ix || !out || strand < 0 || strand > 1) return fail(GSX_ERR_ARG, "bad argument");
    const HostStrand& h = ix->host.st[strand];
    static const uint8_t SYM[4] = {'A', 'C', 'G', 'T'};
    for (uint64_t row = 0; row < h.n; row++) {
        const OccBlock& b = h.blocks[row >> 6];
        out[row] = SYM[block_sym(b.hi, b.lo, (uint32_t)row)];
    }
    for (size_t i = 0; i < h.exc_rows.size(); i++) out[h.exc_rows[i]] = h.exc_sym[i];
    return GSX_OK;
}

extern "C" int gsx_index_export_sa_samples(const gsx_index* ix, int strand, uint32_t* out, uint64_t* n_samples, uint32_t* sa_shift) {
    if (!ix || strand < 0 || strand > 1) return fail(GSX_ERR_ARG, "bad argument");
    const HostStrand& h = ix->host.st[strand];
    if (n_samples) *n_samples = h.sa_samples.size();
    if (sa_shift) *sa_shift = h.sa_shift;
    if (out) memcpy(out, h.sa_samples.data(), h.sa_samples.size() * 4);
    return GSX_OK;
}

// ---------------------------------------------------------------------------------------------------------
// enumerate
// ---------------------------------------------------------------------------------------------------------
// ---- allocation pools -----------------------------------------------------------------------------------------
namespace {
struct Pool {
    std::mutex mu;
    std::multimap<size_t, void*> free_;
    std::map<void*, size_t> capacity;        // pinned host blocks: what each was allocated with (a block may serve a smaller request)
};
Pool& pool_of(int device) { static Pool pools[65]; return pools[device + 1]; }
size_t bucket(size_t bytes) { size_t b = 512; while (b < bytes) b <<= 1; return b; }
}  // namespace

void* gsx::pool_get(int device, size_t bytes) {
    size_t b = bucket(bytes);
    Pool& P = pool_of(device);
    {
        std::lock_guard<std::mutex> g(P.mu);
        // pinned host memory costs half a second per GB to allocate (profiles/r02z_d2h_probe.json) and the result arrays of
        // successive batches straddle bucket boundaries: a free block of up to four times the bucket serves the request
        auto it = device < 0 ? P.free_.lower_bound(b) : P.free_.find(b);
        if (it != P.free_.end() && (device >= 0 || it->first <= 4 * b)) { void* p = it->second; P.free_.erase(it); return p; }
    }
    void* p = nullptr;
    cudaError_t e = device < 0 ? cudaHostAlloc(&p, b, cudaHostAllocDefault) : cudaMalloc(&p, b);
    if (e != cudaSuccess) {                       // give cached blocks back to the driver and retry once
        cudaGetLastError(); pool_trim(device);
        e = device < 0 ? cudaHostAlloc(&p, b, cudaHostAllocDefault) : cudaMalloc(&p, b);
        if (e != cudaSuccess) { cudaGetLastError(); return nullptr; }
    }
    if (device < 0) { std::lock_guard<std::mutex> g(P.mu); P.capacity[p] = b; }
    return p;
}
void gsx::pool_put(int device, void* p, size_t bytes) {
    if (!p) return;
    Pool& P = pool_of(device);
    std::lock_guard<std::mutex> g(P.mu);
    size_t key = bucket(bytes);
    if (device < 0) { auto c = P.capacity.find(p); if (c != P.capacity.end()) key = c->second; }      // (its real size, not the request's)
    P.free_.emplace(key, p);
}
void gsx::pool_trim(int device) {
    Pool& P = pool_of(device);
    std::lock_guard<std::mutex> g(P.mu);
    for (auto& kv : P.free_) { if (device < 0) { cudaFreeHost(kv.second); P.capacity.erase(kv.second); } else cudaFree(kv.second); }
    P.free_.clear();
}

struct DevBufs {
    int device;
    std::vector<std::pair<void*, size_t>> ptrs;
    explicit DevBufs(int dev) : device(dev) {}
    template <class T> T* alloc(size_t n, bool zero = false, cudaStream_t s = 0) {
        size_t b = std::max<size_t>(n, 1) * sizeof(T);
        void* p = pool_get(device, b);
        if (!p) throw CudaError("out of device memory");
        ptrs.emplace_back(p, b);
        if (zero) CK(cudaMemsetAsync(p, 0, b, s));
        return (T*)p;
    }
    void free_one(void* p) { for (auto it = ptrs.begin(); it != ptrs.end(); ++it) if (it->first == p) { pool_put(device, p, it->second); ptrs.erase(it); return; } }
    ~DevBufs() { for (auto& q : ptrs) pool_put(device, q.first, q.second); }
};

// pinned, device-visible words for the small read-backs of a job (gsx_kernels.cu launch_publish), recycled between calls
namespace {
struct Mailbox {
    uint32_t* p = nullptr;
    static std::mutex& mu() { static std::mutex m; return m; }
    static std::vector<uint32_t*>& free_list() { static std::vector<uint32_t*> v; return v; }
    Mailbox() {
        { std::lock_guard<std::mutex> g(mu()); if (!free_list().empty()) { p = free_list().back(); free_list().pop_back(); } }
        if (!p) { void* q = nullptr; if (cudaHostAlloc(&q, 256, cudaHostAllocMapped | cudaHostAllocPortable) != cudaSuccess) { cudaGetLastError(); throw CudaError("cudaHostAlloc (mailbox)"); } p = (uint32_t*)q; }
        memset(p, 0, 256);
    }
    ~Mailbox() { std::lock_guard<std::mutex> g(mu()); free_list().push_back(p); }
};
}  // namespace

static std::mutex g_recs_mu;
static std::vector<std::vector<GuideRec>> g_recs_free;          // record arrays of released results, reused by later calls

int gsx_prepare_guides(const gsx_guide* guides, size_t n, const gsx_params* p, gsx::Prepared& out) {
    if (p->max_bulge_size != 1) return fail(GSX_ERR_ARG, "max_bulge_size must be 1 (the reference hard-wires it: process.hpp:82-87)");
    if (p->mismatches >= (uint32_t)kMaxDist) return fail(GSX_ERR_ARG, "mismatches must be <= 7");
    if (p->rna_bulges > 7 || p->dna_bulges > 7) return fail(GSX_ERR_ARG, "bulge counts must be <= 7");
    if (p->threshold >= kMaxDist) return fail(GSX_ERR_ARG, "threshold must be <= 7");
    if (p->n_alt_pams + 1 > (uint32_t)kMaxPams) return fail(GSX_ERR_ARG, "too many alternative PAMs (max 7)");
    memset(out.pamsets, 0, sizeof out.pamsets);
    std::map<std::string, int> set_of;
    {   // a record array released by an earlier result, if any: fresh multi-megabyte allocations cost more in page faults
        // than the packing itself
        std::lock_guard<std::mutex> lk(g_recs_mu);
        if (!g_recs_free.empty()) { out.recs = std::move(g_recs_free.back()); g_recs_free.pop_back(); }
    }
    out.recs.resize(n);
    std::vector<uint8_t> setid(n);
    const bool bulges = p->rna_bulges || p->dna_bulges;
    uint8_t sym_tab[256], csym_tab[256];                          // symbol code of a character / of its complement
    for (int c = 0; c < 256; c++) { sym_tab[c] = sym_of((char)c); csym_tab[c] = sym_of(complement_char((char)c)); }
    // pass 1 (sequential, light): PAM column values -> PAM sets (process.hpp:51-56)
    size_t set_mp[kMaxPamSets] = {0};
    {
        const char* last_pam = nullptr; int last_set = -1;
        for (size_t i = 0; i < n; i++) {
            const char* pam = guides[i].pam ? guides[i].pam : "";
            if (last_pam && (pam == last_pam || strcmp(pam, last_pam) == 0)) { setid[i] = (uint8_t)last_set; continue; }
            size_t pl = strlen(pam);
            if (pl > (size_t)kMaxPamLen) return fail(GSX_ERR_ARG, "PAM longer than 8");
            auto it = set_of.find(pam);
            if (it == set_of.end()) {
                if (set_of.size() >= (size_t)kMaxPamSets) return fail(GSX_ERR_ARG, "more than 16 distinct PAM column values in one call");
                int id = (int)set_of.size();
                PamSet& ps = out.pamsets[id];
                std::vector<std::string> pams;
                if (pl == 0) pams.push_back("");
                else { for (uint32_t a = 0; a < p->n_alt_pams; a++) pams.push_back(p->alt_pams[a] ? p->alt_pams[a] : ""); pams.push_back(pam); }
                ps.n_pams = (uint8_t)pams.size(); ps.kpam_len = (uint8_t)pl;
                for (size_t k = 0; k < pams.size(); k++) {
                    const std::string& s = pams[k];
                    if (s.size() > (size_t)kMaxPamLen) return fail(GSX_ERR_ARG, "alternative PAM longer than 8");
                    if (s.empty() && pams.size() > 1) return fail(GSX_ERR_ARG, "empty alternative PAM");
                    ps.plen[k] = (uint8_t)s.size();
                    for (size_t j = 0; j < s.size(); j++) {
                        // under iupac_pams a class letter is one character of code SYM_CLS with its members in cmask (complemented in
                        // the default orientation: iupac_complement, not complement_char, which keeps the reference's parity)
                        const char c = p->start ? s[s.size() - 1 - j] : s[j];
                        if (p->iupac_pams && iupac_is_class(c)) { ps.sym[k][j] = SYM_CLS; ps.cmask[k][j] = (uint8_t)iupac_mask(p->start ? c : iupac_complement(c)); }
                        else ps.sym[k][j] = p->start ? sym_of(c) : sym_of(complement_char(c));
                    }
                    set_mp[id] = std::max(set_mp[id], s.size());
                }
                out.max_pams = std::max<uint32_t>(out.max_pams, ps.n_pams);
                it = set_of.emplace(pam, id).first;
            }
            setid[i] = (uint8_t)it->second;
            last_pam = pam; last_set = it->second;
        }
    }
    // pass 2 (parallel over chunks of guides): symbol packing in consumption order (process.hpp:63, index.hpp:214)
    out.gq.resize(n);
    struct Chunk { size_t max_total = 0; uint32_t min_qlen = 255, max_qlen = 0; bool bad_len = false, fast = true; };
    const size_t n_thr = std::max<size_t>(1, std::min<size_t>({(size_t)16, n / 8192, (size_t)std::max(1u, std::thread::hardware_concurrency())}));
    std::vector<Chunk> chunks(n_thr);
    auto work = [&](size_t t) {
        Chunk c;                                                               // (local: the chunk array shares cache lines)
        struct Publish { Chunk& dst; Chunk& src; ~Publish() { dst = src; } } publish{chunks[t], c};
        for (size_t i = n * t / n_thr, e = n * (t + 1) / n_thr; i < e; i++) {
            const char* seq = guides[i].seq ? guides[i].seq : "";
            const size_t sl = strlen(seq);
            if (sl == 0 || sl > (size_t)kMaxQ) { c.bad_len = true; return; }
            GuideRec& r = out.recs[i];
            memset(&r, 0, sizeof r);
            r.qlen = (uint8_t)sl; r.seqlen = (uint8_t)sl; r.pamset = setid[i];
            memcpy(r.seq, seq, sl);
            uint64_t v = (uint64_t)sl << 58; bool acgt = true;
            for (size_t l = 0; l < sl; l++) {
                const uint8_t sy = p->start ? sym_tab[(unsigned char)seq[sl - 1 - l]] : csym_tab[(unsigned char)seq[l]];
                r.q[l] = sy;
                if (sy > 3) acgt = false; else if (l < 29) v |= (uint64_t)sy << (2 * l);
            }
            out.gq[i] = v;
            if (!acgt || sl > 29) c.fast = false;
            c.max_total = std::max(c.max_total, sl + set_mp[r.pamset]);
            c.min_qlen = std::min<uint32_t>(c.min_qlen, (uint32_t)sl); c.max_qlen = std::max<uint32_t>(c.max_qlen, (uint32_t)sl);
        }
    };
    if (n_thr == 1) work(0);
    else { std::vector<std::thread> th; for (size_t t = 0; t < n_thr; t++) th.emplace_back(work, t); for (auto& x : th) x.join(); }
    size_t max_total = 0; bool all_fast = true; out.min_qlen = 255;
    for (const Chunk& c : chunks) {
        if (c.bad_len) return fail(GSX_ERR_ARG, "guide sequence length must be 1..32");
        max_total = std::max(max_total, c.max_total); all_fast = all_fast && c.fast; out.min_qlen = std::min(out.min_qlen, c.min_qlen);
        out.max_qlen = std::max(out.max_qlen, c.max_qlen);
    }
    // PAMs of different lengths inside one set give match strings of different lengths: only the left-aligned (wide) key
    // orders those as std::string does
    bool same_plen = true;
    for (size_t k = 0; k < set_of.size(); k++) for (int j = 1; j < out.pamsets[k].n_pams; j++) same_plen = same_plen && out.pamsets[k].plen[j] == out.pamsets[k].plen[0];
    out.wide = bulges || max_total > 27 || !same_plen;
    if (max_total + p->dna_bulges > 32) return fail(GSX_ERR_ARG, "guide + PAM + DNA bulges longer than 32 characters");
    // fast path: no bulges, the same PAM list for every guide (alternative PAMs = one search pass each), ACGT-only guides of
    // at most 29 nt
    out.fast_ok = !out.wide && set_of.size() == 1 && n > 0 && all_fast;
    // bulges: the same batch with every guide replaced by its edited guides (gsx_core.h variant_rewrite), if those are few
    // enough to be worth it and still fit the narrow keys
    out.variant_ok = bulges && set_of.size() == 1 && n > 0 && all_fast && same_plen && max_total + p->dna_bulges <= 27 &&
                     out.max_qlen + p->dna_bulges <= 29 && p->rna_bulges + p->dna_bulges <= 4 && env_int("GSX_VARIANTS", 1) &&
                     bulge_variant_count(out.max_qlen, p->rna_bulges, p->dna_bulges) <= (uint64_t)env_int("GSX_VARIANTS_MAX", 8192);
    if (out.fast_ok || out.variant_ok) {
        const PamSet& ps = out.pamsets[0];
        out.n_fast_pams = ps.n_pams;
        for (uint32_t k = 0; k < ps.n_pams; k++) {
            out.plens[k] = ps.plen[k]; out.pampacks[k] = 0; out.pammasks[k] = 0;
            for (uint32_t j = 0; j < ps.plen[k]; j++) {
                out.pampacks[k] |= (uint32_t)ps.sym[k][j] << (3 * j);
                out.pammasks[k] |= (uint32_t)ps.cmask[k][j] << (4 * j);
            }
        }
        out.plen = out.plens[0]; out.pampack = out.pampacks[0]; out.pammask = out.pammasks[0];
    }
    return GSX_OK;
}

// Small batches on the general kernel: a (guide, strand) task occupies one warp, so a few hundred guides would leave most
// of the grid idle while a bulge search runs for seconds.  The roots are therefore expanded on the host, breadth first and
// through the kernels' own node arithmetic (gsx_core.h make_child over the host copy of the blocks), until there are enough
// nodes for every warp; the kernel then takes those nodes as its tasks.  Same tree, same matches.
template <bool WIDE>
static std::vector<Node> expand_roots(const gsx_index* ix, const Prepared& prep, size_t g0, uint32_t n, uint32_t M, uint32_t R, uint32_t D,
                                      size_t want, uint32_t max_depth) {
    const DevStrand st[2] = {host_view(ix->host.st[0]), host_view(ix->host.st[1])};
    std::vector<Node> cur;
    for (uint32_t t = 0; t < 2 * n; t++) { Node r{}; r.sp = 0; r.ep = st[t & 1].n - 1; r.task = t; cur.push_back(r); }
    for (uint32_t depth = 0; depth < max_depth && cur.size() < want; depth++) {
        std::vector<Node> nxt; nxt.reserve(cur.size() * 4);
        for (const Node& nd : cur) {
            const DevStrand& s = st[nd.task & 1];
            const GuideRec& g = prep.recs[g0 + (nd.task >> 1)];
            ExpandCtx cx{&s, &g, &prep.pamsets[g.pamset], M, R, D};
            uint32_t os[4], oe[4];
            const OccBlock& b0 = s.blocks[nd.sp >> 6]; const OccBlock& b1 = s.blocks[(nd.ep + 1) >> 6];
            block_occ(s, b0.cnt, b0.hi, b0.lo, nd.sp, os); block_occ(s, b1.cnt, b1.hi, b1.lo, nd.ep + 1, oe);
            for (int cand = 0; cand < CAND_END; cand++) {
                if (!WIDE && cand > CAND_FORK) break;
                Node ch; bool emit;
                if (!make_child<WIDE>(cand, nd, cx, os, oe, ch, emit)) continue;
                if (emit) return cur;            // a finished alignment this close to the root (very short guide): keep the last complete level
                nxt.push_back(ch);
            }
        }
        cur.swap(nxt);
    }
    return cur;
}

// ---- the search plan ----------------------------------------------------------------------------------------------------------
static constexpr uint32_t kSplitHalf = 10;          // the two-part sweep cuts its 20-nt guides here
static constexpr int kUnset = INT_MIN;              // a knob that is not set
SearchPlan gsx::plan_search(const Prepared& prep, const gsx_params& p, const IndexShape& ix, uint32_t n) {
    SearchPlan pl;
    const uint32_t L = ix.ftab_L[0];
    pl.variant_general[0] = env_int("GSX_SEARCH_VARIANT", 0); pl.variant_general[1] = env_int("GSX_SEARCH_VARIANT_WIDE", 0);
    pl.variant_fast = env_int("GSX_FAST_VARIANT", ix.lines ? 1 : 0);
    // fast path (search_fast_kernel) when the batch and the index allow it; GSX_FORCE_GENERAL=1 keeps the general kernel
    // (an index whose only non-ACGT BWT row is the sentinel runs the plain kernels; genomes with N / IUPAC characters -- every
    // real assembly -- run search_fast_kernel<..., EXC> behind the same sweep: 4.75 M guides/s against 80 k on the general kernel
    // at 3.1 Gb with 300 runs of N, output identical to the CPU arm's, profiles/r02a_session_3100mb.jsonl; GSX_FAST_ON_N=0 turns it off)
    pl.exc = !ix.plain && env_int("GSX_FAST_ON_N", 1) != 0 && pl.variant_fast == 1 && ix.exc_map;
    pl.use_fast = (prep.fast_ok || prep.variant_ok) && !env_int("GSX_FORCE_GENERAL", 0) && n < (1u << 23) && (ix.plain || pl.exc);
    // bulges: the search runs over the guides' edited forms (gsx_core.h variant_rewrite), in chunks, on the same kernels
    pl.use_variants = pl.use_fast && prep.variant_ok;
    // The specialised kernels read the packed guides (8 bytes each) only; the 80-byte records are needed from the locate stage
    // on.  Their upload (pageable host memory: the call blocks the host) is issued on a second stream AFTER the first search
    // launch, so that it runs under the search instead of in front of it.
    pl.late_guides = pl.use_fast && !pl.use_variants;
    const bool wide = prep.wide;
    pl.search_warps = pl.use_fast ? search_fast_grid_warps(pl.variant_fast, ix.sm_count) : search_grid_warps(wide, pl.variant_general[wide], ix.sm_count);
    pl.threshold_warps = pl.use_fast ? pl.search_warps : search_grid_warps(false, pl.variant_general[0], ix.sm_count);
    if (pl.use_fast) {
        // L2 residency hint: intervals wide enough that all such blocks of both strands fit the L2 budget
        // (a level-d interval end costs one 128-byte line; lines touched down to level D ~ 2.7 * 4^D per strand)
        const double l2_bytes = (double)env_int("GSX_L2_PIN_MB", 64) * 1e6;
        const double w = l2_bytes > 0 ? (double)ix.rows * 2.0 * 2.7 * 128.0 / l2_bytes : 4.0e9;
        pl.pin_width = w >= 4.0e9 ? 0xFFFFFFFFu : (uint32_t)std::max(256.0, w);
    }
    // slice-major front end (sweep_kernel) for large batches: needs the jump table and the look-ahead lines
    pl.ftab_L = L; pl.sweep_variant_set = env_int("GSX_SWEEP_VARIANT", kUnset); pl.load_mode = (uint32_t)env_int("GSX_SWEEP_LOAD", 2);
    if (pl.use_fast && L >= 6 && ix.ftab_L[1] == L && ix.sum0 && env_int("GSX_SWEEP", 1)) {
        const double per_strand = 40.0 * std::pow(4.0, (double)L);                     // sum0 + the part of sum1 that is touched
        const double target = (double)env_int("GSX_SWEEP_SLICE_MB", 12) * 1e6;
        uint32_t sb = 1; while (sb < L - 3 && per_strand / std::pow(4.0, (double)sb) > target) sb++;
        if (env_int("GSX_SWEEP_SB", 0) > 0) sb = (uint32_t)env_int("GSX_SWEEP_SB", 0);
        pl.sweep_width = sb >= 1 && sb + 3 <= L ? sb : 0; pl.sweep_min = (uint32_t)env_int("GSX_SWEEP_MIN", 8192);
    }
    pl.search_sb = pl.use_variants ? 0u : pl.sweep_sb(n, prep.min_qlen, std::max<uint32_t>(p.mismatches, p.threshold > 0 ? (uint32_t)p.threshold : 0u));
    if (p.threshold > 0) pl.threshold_sb = pl.sweep_sb(n, prep.min_qlen, (uint32_t)p.threshold);
    pl.combos = pl.use_fast && L && !pl.search_sb; pl.threshold_combos = p.threshold > 0 && pl.use_fast && L && !pl.threshold_sb;
    // Two-part enumeration (sweep_split_kernel, GSX_SPLIT=0 turns it off): 20-nt guides, one PAM of the form N + two concrete
    // characters, at most 3 mismatches, an index without N, no --start, no threshold pass, and a jump table deep enough to hold
    // both capped halves (13 characters: the PAM and the proximal half of the PAM-first form; with fewer, that form would hand the
    // tree search alignments with two proximal mismatches only for the re-anchoring to drop them).  Per guide and strand a quarter
    // of the summary sectors of the plain sweep.  A class PAM character (code 6) is not concrete, so class PAMs keep the plain sweep.
    pl.split = pl.search_sb != 0 && !pl.use_variants && p.threshold <= 0 && !p.start && prep.n_fast_pams == 1 && prep.plen == 3 &&
               (prep.pampack & 7u) == 4u && ((prep.pampack >> 3) & 7u) < 4u && ((prep.pampack >> 6) & 7u) < 4u &&
               prep.min_qlen == 2 * kSplitHalf && prep.max_qlen == 2 * kSplitHalf && p.mismatches <= kSplitMaxM && ix.plain &&
               L >= prep.plen + kSplitHalf && n < (1u << 22) && env_int("GSX_SPLIT", 1) != 0;
    if (pl.split) {
        // slices one character wider than the plain sweep's: a quarter of the patterns per guide, so four times the slice keeps the
        // patterns per work unit up (3.1 Gb, 200 k guides, one B200: sweep 13.0 ms at sb = 4 against 15.9 at 5 and 15.7 at 3,
        // profiles/r03a_split_ab_3100mb_200k.jsonl)
        pl.split_sb = env_int("GSX_SPLIT_SB", 0) > 0 ? (uint32_t)env_int("GSX_SPLIT_SB", 0) : (pl.search_sb > 1 ? pl.search_sb - 1 : pl.search_sb);
        pl.split_ctas = env_int("GSX_SPLIT_CTAS", 6);
    }
    // alternative PAMs (process.hpp:51-56): the searches of the PAMs are independent and their matches are collected in
    // the same per-guide sets, so each PAM gets its own pass over the same arenas; only the work counters start over
    // Default (GSX_FUSED_PAMS=0 keeps one pass per PAM; m = 4 with NGG + NAG at 3.1 Gb: 232 k against 142 k guides/s, same text): the PAMs in
    // ONE pass -- search with the filter PAM, keep the alignments whose PAM characters spell a real PAM (gsx_core.h fused_pam_ok)
    pl.fuse_pams = prep.n_fast_pams > 1 && pl.variant_fast == 1 && env_int("GSX_FUSED_PAMS", 1) != 0;
    if (!pl.use_fast) {
        const int gw = search_grid_warps(wide, pl.variant_general[wide], ix.sm_count);
        if (gw > 0 && (uint64_t)2 * n < (uint64_t)4 * gw) pl.expand_roots = (size_t)8 * gw;          // fewer tasks than the grid can keep busy
    }
    // seed queue of the sweep: 12 survivors per guide measured at m = 3 on 3.1 Gb (two orders of magnitude more at m = 4);
    // sized with a wide margin, never beyond the 32-bit slot numbers the kernels use; an overflow is retried with 4x the room
    const uint64_t queue_set = (uint64_t)std::max(env_int("GSX_QUEUE_CAP", 0), 0);
    pl.queue_cap = queue_set ? queue_set : std::min<uint64_t>(std::max<uint64_t>((uint64_t)n * (p.mismatches >= 4 ? 1024 : 256), 1u << 20), 1ull << 30);
    // Match arena: an overflow costs a second run of the whole search, so the first size has to be right.  Expected matches per
    // guide on a genome without structure = 2 strands x rows x (substitution patterns within the budget) / 4^length x the fraction
    // of sites a PAM list accepts: 11 at 3 mismatches / NGG on 3.1 Gb, 300 at 4 mismatches with NGG + NAG (the size round 1 got
    // wrong: n x 48 -- every such call searched twice).  The job raises it to what earlier calls on the index needed.
    pl.match_per_guide = wide ? 2048.0 : 48.0;
    if (!wide) {
        const double ql = (double)std::max<uint32_t>(prep.min_qlen, 1);
        double patterns = 0, c = 1;                                           // sum over j <= M of C(q, j) 3^j
        for (uint32_t j = 0; j <= p.mismatches && j <= prep.min_qlen; j++) { patterns += c; c = c * 3.0 * (ql - j) / (j + 1.0); }
        double pam_frac = 0;
        for (int ps = 0; ps < kMaxPamSets; ps++) {
            double f = 0;
            const PamSet& P = prep.pamsets[ps];
            for (int k = 0; k < P.n_pams; k++) {
                double g1 = 1;                                                // a class character passes |class| / 4 of the sites
                for (int j = 0; j < P.plen[k]; j++) g1 *= P.sym[k][j] == SYM_CLS ? 0.25 * popc64(P.cmask[k][j]) : P.sym[k][j] != SYM_N ? 0.25 : 1.0;
                f += g1;
            }
            pam_frac = std::max(pam_frac, std::min(1.0, f));
        }
        const double expect = 2.0 * (double)ix.rows * patterns / std::pow(4.0, ql) * pam_frac;
        pl.match_per_guide = std::max(pl.match_per_guide, 1.5 * expect + 8.0);
    }
    pl.match_cap_set = (uint64_t)std::max(env_int("GSX_MATCH_CAP", 0), 0);      // tests: force the retry path
    const uint32_t spill_set = (uint32_t)std::max(env_int("GSX_SPILL_CAP", 0), 0);
    pl.spill_cap = spill_set ? spill_set : (wide && !pl.use_variants) ? 8192 : 2048;
    if (pl.use_variants) {
        const uint32_t R = p.rna_bulges, D = p.dna_bulges;
        pl.chunk = (uint32_t)std::min<int64_t>(std::max<int64_t>(env_int("GSX_VARIANT_CHUNK", 262144), 1), (1 << 22));
        // the sweep skips patterns that substitute an inserted position (GSX_FORCED_SWEEP=0: it tests them and the rewrite drops their
        // matches; 11 % fewer seeds, 1.4 % less search time at 3.1 Gb)
        pl.fmask = env_int("GSX_FORCED_SWEEP", 1) != 0;
        pl.edited_qmin = prep.min_qlen > R ? prep.min_qlen - R : 0; pl.edited_qmax = prep.max_qlen + D;
        pl.chunk_queue_cap = queue_set ? queue_set : std::max<uint64_t>((uint64_t)pl.chunk * 256, 1u << 20);
        pl.chunk_match_cap = std::max<uint64_t>((uint64_t)pl.chunk * 48, 1u << 18);
        pl.edited_match_cap = std::max<uint64_t>(1u << 18, std::min<uint64_t>((uint64_t)n * bulge_variant_count(prep.max_qlen, R, D) * 12, 1u << 26));
        if (pl.match_cap_set) pl.chunk_match_cap = pl.edited_match_cap = pl.match_cap_set;
    }
    // match ordering (GSX_ORDER: 0 warp per guide, 1 CTA per guide, 2 radix sort) and specificity (GSX_SPEC_WARP) by default follow
    // the matches and hits per guide, known after the search
    pl.order_probe = !env_int("GSX_ORDER", 0) && !env_int("GSX_ORDER_CTA", 0);
    pl.order_mode = env_int("GSX_ORDER", env_int("GSX_ORDER_CTA", 0) ? 1 : kUnset); pl.spec_warp = env_int("GSX_SPEC_WARP", kUnset);
    return pl;
}

uint32_t SearchPlan::sweep_sb(uint32_t ng, uint32_t min_qlen, uint32_t M) const {
    if (!sweep_width || ng < sweep_min || min_qlen < ftab_L || M > 4) return 0;
    return 2.0 * std::pow(4.0, (double)sweep_width) * ((ng + 31) / 32) * 8.0 >= 4.0e9 ? 0 : sweep_width;      // (32-bit work units)
}

// sweep_lean_kernel (variants 10-12) where its compiled loops cover the batch: at most 4 mismatches, every guide length of the
// batch giving one of its plane layouts; sweep_kernel (variant 2) otherwise.  Measured at 3.1 Gb
// (profiles/r02c_session_3100mb_sweep_lean3.jsonl): six CTAs per SM (variant 12) for plain batches of at most 3 mismatches --
// 24.0 ms per 200 k guides against 36.6 for sweep_kernel --, five (variant 11) for 4 mismatches and for the edited guides of a
// bulge search
int SearchPlan::sweep_variant(uint32_t M, uint32_t qmin, uint32_t qmax, uint32_t plen, uint32_t pampack) const {
    const int sv = sweep_variant_set != kUnset ? sweep_variant_set : (M <= 3 && !use_variants) ? 12 : 11;
    bool lean = M <= 4;
    for (uint32_t ql = qmin; lean && ql <= qmax; ql++) lean = sweep_shape_of(sweep_codes((uint64_t)ql << 58, ftab_L, plen, pampack)) >= 0;
    return sv >= 10 && !lean ? 2 : sv;
}

static IndexShape shape_of(const DeviceIndex& di) {
    const DevStrand &a = di.st[0].d, &b = di.st[1].d;
    return IndexShape{a.n_exc == 1 && b.n_exc == 1 && a.n_nrows == 0 && b.n_nrows == 0, a.lines != nullptr, di.st[0].exc_map && di.st[1].exc_map,
                      {a.ftab_L, b.ftab_L}, a.sum0 && b.sum0, a.n, di.sm_count};
}

// ---- the device job -----------------------------------------------------------------------------------------------------------
// streams and events of one device job: released on every path out of run_device_job (errors included); in-flight copies are
// waited for first, because the buffers they touch go back to the allocation pools right after
enum JobEvent { kSearchBegin, kSearchEnd, kArrangeEnd, kLocateEnd, kScoreEnd, kCopyEnd, kSweepBegin, kSweepEnd, kJobEvents };
struct JobStreams {
    cudaStream_t s = nullptr, s2 = nullptr;
    cudaEvent_t ev[kJobEvents] = {}, ev_guides = nullptr;
    ~JobStreams() {
        if (s) cudaStreamSynchronize(s);
        if (s2) cudaStreamSynchronize(s2);
        for (auto& e : ev) if (e) cudaEventDestroy(e);
        if (ev_guides) cudaEventDestroy(ev_guides);
        if (s) cudaStreamDestroy(s);
        if (s2) cudaStreamDestroy(s2);
        cudaGetLastError();                                      // (a failed job must not leave a sticky error code for the next call's first check)
    }
};

struct DeviceJob {
    const gsx_index* ix = nullptr; int slot = 0;
    const Prepared* prep = nullptr; const gsx_params* p = nullptr;
    size_t g0 = 0, g1 = 0;
    HostArrays out; gsx_counters ctr{};
    int status = GSX_OK; std::string err;
    uint32_t want = kWantAll;            // per-hit arrays to bring to the host (gsx_host.h)
};

// the sweep's state: xor table (of the last M and slice width), per-guide filter masks, seed queue
struct SweepState {
    uint32_t* xtab = nullptr; uint32_t xtab_M = ~0u, xtab_sb = 0, n_xtab = 0; SweepPlan plan{};
    uint32_t* gtab = nullptr; size_t gtab_cap = 0; SeedNode* queue = nullptr; uint64_t queue_cap = 0;
};
// the two-part sweep's own state: its xor table, the PAM-first queries, their seed queue and match arena, and their counters
struct SplitState {
    uint32_t* xtab = nullptr; uint32_t n_xtab = 0; SplitPlan plan{};
    uint64_t* gq2 = nullptr; uint32_t* nmatch2 = nullptr; SeedNode* queue2 = nullptr; uint64_t queue2_cap = 0;
    MatchRec* matches2 = nullptr; uint64_t matches2_cap = 0; bool ran = false;
    uint32_t* ctrs2 = nullptr;           // [0] form-1 seed count [1] task counter [2] form-1 match count
};
// a match arena search_until_fits grows: records, capacity, and the error when it would pass 2^31 records
struct MatchArena { MatchRec* p; uint64_t cap; const char* too_many; };
#define LAUNCH(call) do { CK(call); n_launches++; } while (0)

// One device job's state; run_device_job calls its stages in order.
struct DeviceRun {
    DeviceJob& job; const DeviceIndex& di; const Prepared& prep; const gsx_params& p;
    const uint32_t n, n_dist;
    const SearchPlan plan;
    const uint64_t learn_key;            // index of learned_matches_per_guide: the option set
    DevBufs B;
    Mailbox mbox;                        // (declared before the streams: they are drained before it goes back to the free list)
    JobStreams js;                       // (declared after the buffer holder: destroyed -- synchronised -- before it)
    cudaStream_t &s = js.s, &s2 = js.s2;
    // Calls from several host threads (the reference's own worker threads, or gsx_enumerate_start) take turns on a device from the
    // first search launch to the last result copy (gsx::device_turn).
    std::unique_lock<std::mutex> turn;
    uint64_t n_launches = 0; bool guides_up = false;
    GuideRec* d_guides = nullptr; PamSet* d_pamsets = nullptr; uint32_t* d_nmatch = nullptr; uint8_t* d_dropped = nullptr; unsigned long long* d_stats = nullptr;
    uint32_t* d_ctrs = nullptr;          // [0] task counter [1] match count [2] error flag [3] seed queue count [4] sweep work units [5] final matches
    SearchArgs a{};                      // what every search launch of the job starts from
    SweepState sw; SplitState sp;
    uint32_t qmin = 0, qmax = 0;         // guide lengths of the batch the fast kernels see (edited guides: - R .. + D)
    MatchRec* d_matches = nullptr; uint32_t n_matches = 0, n_seeds = 0; bool use_sweep = false;
    uint32_t *d_moff = nullptr, *d_sorted = nullptr, *d_sorted_off = nullptr, *d_nhits = nullptr, *d_hoff = nullptr, *d_cbd = nullptr;
    uint32_t *d_hit_match = nullptr, *d_hit_row = nullptr, nh = 0;
    LocateArgs L{}; SpecArgs S{}; unsigned long long stats[8] = {};

    explicit DeviceRun(DeviceJob& j)
        : job(j), di(j.ix->dev[j.slot]), prep(*j.prep), p(*j.p), n((uint32_t)(j.g1 - j.g0)), n_dist(j.p->mismatches + 1),
          plan(plan_search(prep, p, shape_of(di), n)),
          learn_key((uint64_t)p.mismatches | ((uint64_t)prep.n_fast_pams << 8) | ((uint64_t)p.rna_bulges << 16) | ((uint64_t)p.dna_bulges << 24) |
                    ((uint64_t)prep.min_qlen << 32) | ((uint64_t)(prep.wide ? 1 : 0) << 40)), B(di.device) {}
    // the first words of d_ctrs, read on the host without touching the copy engine
    void read_ctrs(uint32_t* h, uint32_t n_words, const uint32_t* d_src) {
        CK(launch_publish(d_src, n_words, mbox.p, s)); CK(cudaStreamSynchronize(s));
        for (uint32_t i = 0; i < n_words; i++) h[i] = mbox.p[i];
    }
    void upload_guides(cudaStream_t st) {
        if (guides_up) return;
        const auto t0 = std::chrono::steady_clock::now();
        CK(cudaMemcpyAsync(d_guides, prep.recs.data() + job.g0, (size_t)n * sizeof(GuideRec), cudaMemcpyHostToDevice, st));
        CK(cudaEventRecord(js.ev_guides, st)); guides_up = true;
        job.ctr.ms_h2d += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    }
    // every way to substitute at most M of the jump table's characters but the last two (search_fast_kernel without a sweep)
    void upload_combos(SearchArgs& m, uint32_t M) {
        const std::vector<uint64_t> cb = ftab_combos(plan.ftab_L - 2, M);
        uint64_t* d_cb = B.alloc<uint64_t>(cb.size());
        CK(cudaMemcpyAsync(d_cb, cb.data(), cb.size() * 8, cudaMemcpyHostToDevice, s)); CK(cudaStreamSynchronize(s));
        m.combos = d_cb; m.n_combos = (uint32_t)cb.size();
    }
    // streams, result arrays, the first uploads; false when the batch is empty.  Ends by taking the device's turn.
    bool setup() {
        CK(cudaStreamCreate(&js.s)); CK(cudaStreamCreate(&js.s2));
        for (auto& e : js.ev) CK(cudaEventCreate(&e));
        CK(cudaEventCreateWithFlags(&js.ev_guides, cudaEventDisableTiming));
        HostArrays& H = job.out; H.n_guides = n;
        H.dropped = H.alloc<uint8_t>(n); H.n_hits_of = H.alloc<uint32_t>(n); H.hoff = H.alloc<uint32_t>(n + 1);
        H.specificity = H.alloc<float>(n); H.perfect = H.alloc<uint8_t>(n); H.cbd = H.alloc<uint32_t>((size_t)n * n_dist);
        if (n == 0) { H.hoff[0] = 0; return false; }
        d_guides = B.alloc<GuideRec>(n); d_pamsets = B.alloc<PamSet>(kMaxPamSets);
        const auto t_h2d0 = std::chrono::steady_clock::now();
        CK(cudaMemcpyAsync(d_pamsets, prep.pamsets, sizeof(prep.pamsets), cudaMemcpyHostToDevice, s));
        job.ctr.ms_h2d = 0;
        if (!plan.late_guides) upload_guides(s);
        d_nmatch = B.alloc<uint32_t>(n + 1, true, s); d_dropped = B.alloc<uint8_t>(n, true, s);
        d_ctrs = B.alloc<uint32_t>(8, true, s); d_stats = B.alloc<unsigned long long>(8, true, s);
        a.st[0] = di.st[0].d; a.st[1] = di.st[1].d; a.guides = d_guides; a.pamsets = d_pamsets;
        a.task_counter = d_ctrs + 0; a.match_count = d_ctrs + 1; a.error_flag = d_ctrs + 2; a.stats = d_stats;
        a.guide_nmatch = d_nmatch; a.max_iters = 1u << 28; a.max_pams = prep.max_pams; a.p.n_tasks = 2 * n;
        if (plan.use_fast) {
            uint64_t* d_gq = B.alloc<uint64_t>(n);
            CK(cudaMemcpyAsync(d_gq, prep.gq.data() + job.g0, (size_t)n * 8, cudaMemcpyHostToDevice, s));
            if (plan.late_guides) job.ctr.ms_h2d += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_h2d0).count();
            a.gq = d_gq; a.pampack = prep.pampack; a.pammask = prep.pammask; a.plen = prep.plen;
            a.exc = plan.exc ? 1u : 0u; a.exc_map[0] = (const uint32_t*)di.st[0].exc_map; a.exc_map[1] = (const uint32_t*)di.st[1].exc_map;
            a.pin_width = plan.pin_width; a.combos = nullptr; a.n_combos = 0;
        }
        if (plan.split) sp.ctrs2 = B.alloc<uint32_t>(4, true, s);
        sw.queue_cap = plan.queue_cap; qmin = prep.min_qlen; qmax = prep.max_qlen; use_sweep = plan.search_sb != 0;
        turn = gsx::device_turn(di.device);
        CK(cudaEventRecord(js.ev[kSearchBegin], s));
        return true;
    }
    // One search, run until its arenas hold everything it finds.  Each attempt gets a spill stack for the grid, runs `launch` (the
    // caller's counter resets and launches) and reads d_ctrs[0..3] back into h.  On an overflow the arenas grow -- seed queue x4,
    // match arena to max(2x, 1.25x what the search asked for), spill stack x4 -- and the search runs again, at most 12 times more.
    // The grown sizes stay with the caller for its later searches.
    template <class F> void search_until_fits(int warps, uint32_t spill_words, uint32_t& spill_cap, MatchArena* arena, uint32_t h[4], F&& launch) {
        for (int attempt = 0;; attempt++) {
            if (attempt > 12) throw std::runtime_error("search arenas keep overflowing");
            if (warps <= 0) throw std::runtime_error("unknown search kernel variant");
            uint32_t* d_spill = B.alloc<uint32_t>((size_t)warps * spill_cap * spill_words);
            launch(d_spill);
            read_ctrs(h, 4, d_ctrs); n_launches++;
            B.free_one(d_spill);
            if (h[2] & GSX_KERR_WATCHDOG) throw std::runtime_error("search kernel watchdog tripped");
            if (h[2] & GSX_KERR_REANCHOR) throw std::runtime_error("two-part search: a PAM-first match has no interval in the other index");
            if (!(h[2] & (GSX_KERR_MATCH_OVERFLOW | GSX_KERR_SPILL_OVERFLOW | GSX_KERR_QUEUE_OVERFLOW))) return;
            if (h[2] & GSX_KERR_QUEUE_OVERFLOW) { B.free_one(sw.queue); sw.queue = nullptr; sw.queue_cap *= 4; }
            if (sw.queue_cap >= (1ull << 32)) throw std::runtime_error("seed queue keeps overflowing");
            if ((h[2] & GSX_KERR_MATCH_OVERFLOW) && arena) {
                B.free_one(arena->p); arena->cap = std::max<uint64_t>(arena->cap * 2, (uint64_t)h[1] + (h[1] >> 2));
                if (arena->cap > (1ull << 31)) throw std::runtime_error(arena->too_many);
                arena->p = B.alloc<MatchRec>(arena->cap);
            }
            if (h[2] & GSX_KERR_SPILL_OVERFLOW) spill_cap *= 4;
        }
    }
    // threshold prefilter (process.hpp:66-76): mismatch-only counting search, guide dropped if > 1 site
    void threshold_pass() {
        unsigned long long* d_gcount = B.alloc<unsigned long long>(n, true, s);
        SearchArgs base = a;
        if (plan.threshold_combos) upload_combos(base, (uint32_t)p.threshold);
        uint32_t spill_cap = 4096, h[4];
        search_until_fits(plan.threshold_warps, 6, spill_cap, nullptr, h, [&](uint32_t* d_spill) {           // (counting: no match arena)
            CK(cudaMemsetAsync(d_ctrs, 0, 8 * sizeof(uint32_t), s));
            CK(cudaMemsetAsync(d_gcount, 0, (size_t)n * 8, s));
            SearchArgs c = base; c.p.M = (uint32_t)p.threshold; c.p.R = c.p.D = 0; c.p.counting = 1; c.p.match_cap = 0; c.p.spill_cap = spill_cap;
            c.guide_count = d_gcount; c.spill = d_spill; c.skip = nullptr; c.matches = nullptr;
            if (plan.use_fast) run_fast_all_pams(c, n, plan.threshold_sb, nullptr);
            else LAUNCH(launch_search(c, false, plan.variant_general[0], di.sm_count, s, nullptr));
            upload_guides(s2);
        });
        LAUNCH(launch_threshold(d_gcount, d_dropped, n, s));
        unsigned long long zero[8] = {0}; CK(cudaMemcpyAsync(d_stats, zero, sizeof zero, cudaMemcpyHostToDevice, s));
    }
    // the main search: the batch or its edited guides; then what it needed per guide is remembered for the next call
    void search() {
        if (plan.combos) upload_combos(a, p.mismatches);
        if (plan.use_variants) search_edited(); else search_batch();
        CK(cudaEventRecord(js.ev[kSearchEnd], s));
        std::lock_guard<std::mutex> lk(job.ix->learn_mu);
        double& v = job.ix->learned_matches_per_guide[learn_key];
        v = std::max(v * 0.9, (double)n_matches / (double)n);                  // (decays, so that one odd batch does not inflate the arenas for good)
    }
    // all n guides in one search: sweep, two-part sweep, jump-table combos or the general kernel
    void search_batch() {
        const bool wide = prep.wide;
        double per_guide = plan.match_per_guide;                             // raised to what earlier calls on the index needed
        {
            std::lock_guard<std::mutex> lk(job.ix->learn_mu);
            auto it = job.ix->learned_matches_per_guide.find(learn_key);
            if (it != job.ix->learned_matches_per_guide.end()) per_guide = std::max(per_guide, 1.25 * it->second);
        }
        const uint64_t cap = std::min<uint64_t>(std::max<uint64_t>((uint64_t)((double)n * per_guide), 1u << 18), 1u << 27);
        MatchArena out{nullptr, plan.match_cap_set ? plan.match_cap_set : cap, "more than 2^31 matches in one batch; lower the batch size"};
        uint32_t spill_cap = plan.spill_cap;
        Node* d_gseeds = nullptr; uint32_t n_gseeds = 0;
        if (plan.expand_roots) {
            const std::vector<Node> gs = wide ? expand_roots<true>(job.ix, prep, job.g0, n, p.mismatches, p.rna_bulges, p.dna_bulges, plan.expand_roots, 6)
                                              : expand_roots<false>(job.ix, prep, job.g0, n, p.mismatches, p.rna_bulges, p.dna_bulges, plan.expand_roots, 6);
            if (gs.size() > (size_t)2 * n) {
                d_gseeds = B.alloc<Node>(gs.size()); n_gseeds = (uint32_t)gs.size();
                CK(cudaMemcpyAsync(d_gseeds, gs.data(), gs.size() * sizeof(Node), cudaMemcpyHostToDevice, s)); CK(cudaStreamSynchronize(s));
            }
        }
        out.p = B.alloc<MatchRec>(out.cap);
        uint32_t h[4];
        search_until_fits(plan.search_warps, wide ? 8 : 6, spill_cap, &out, h, [&](uint32_t* d_spill) {
            CK(cudaMemsetAsync(d_ctrs, 0, 8 * sizeof(uint32_t), s));
            CK(cudaMemsetAsync(d_nmatch, 0, (size_t)(n + 1) * 4, s));
            CK(cudaMemsetAsync(d_stats, 0, 8 * sizeof(unsigned long long), s));
            SearchArgs m = a; m.p.M = p.mismatches; m.p.R = p.rna_bulges; m.p.D = p.dna_bulges; m.p.counting = 0;
            m.p.match_cap = (uint32_t)out.cap; m.p.spill_cap = spill_cap; m.spill = d_spill; m.matches = out.p;
            m.skip = p.threshold > 0 ? d_dropped : nullptr;
            m.gseeds = d_gseeds; m.n_gseeds = n_gseeds;
            CK(cudaEventRecord(js.ev[kSweepBegin], s));
            if (plan.use_fast) run_fast_all_pams(m, n, plan.search_sb, js.ev[kSweepEnd]);
            else { CK(cudaEventRecord(js.ev[kSweepEnd], s)); LAUNCH(launch_search(m, wide, plan.variant_general[wide], di.sm_count, s, nullptr)); }
            upload_guides(s2);
        });
        d_matches = out.p; n_matches = h[1]; n_seeds = use_sweep ? h[3] : 0;
        if (sp.ran) { uint32_t h1; read_ctrs(&h1, 1, sp.ctrs2); n_seeds += h1; n_launches++; }
    }
    // bulges as edited guides: chunks of guides whose edited forms fill one launch of the specialised kernels.  Each chunk's matches
    // are rewritten into the batch's arena; d_nmatch and d_stats add up over the chunks.
    void search_edited() {
        const uint32_t R = p.rna_bulges, D = p.dna_bulges;
        std::vector<uint32_t> descs, doff(kMaxQ + 2, 0), dcnt(kMaxQ + 2, 0);
        for (uint32_t ql = prep.min_qlen; ql <= prep.max_qlen; ql++) {
            const std::vector<uint32_t> v = bulge_variants(ql, R, D);
            doff[ql] = (uint32_t)descs.size(); dcnt[ql] = (uint32_t)v.size(); descs.insert(descs.end(), v.begin(), v.end());
        }
        uint32_t* d_descs = B.alloc<uint32_t>(descs.size()); uint32_t* d_doff = B.alloc<uint32_t>(doff.size());
        CK(cudaMemcpyAsync(d_descs, descs.data(), descs.size() * 4, cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(d_doff, doff.data(), doff.size() * 4, cudaMemcpyHostToDevice, s));
        std::vector<uint8_t> h_dropped(n, 0);
        if (p.threshold > 0) CK(cudaMemcpyAsync(h_dropped.data(), d_dropped, n, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        const uint32_t chunk_v = plan.chunk;
        qmin = plan.edited_qmin; qmax = plan.edited_qmax;
        if (sw.queue) { B.free_one(sw.queue); sw.queue = nullptr; }               // (sized by the threshold pass)
        sw.queue_cap = plan.chunk_queue_cap;
        uint64_t match_cap = plan.edited_match_cap;
        uint32_t spill_cap = plan.spill_cap;
        uint64_t* d_vq = B.alloc<uint64_t>(chunk_v + 1); uint32_t* d_vdesc = B.alloc<uint32_t>(chunk_v + 1); uint32_t* d_vguide = B.alloc<uint32_t>(chunk_v + 1);
        uint32_t* d_vnmatch = B.alloc<uint32_t>(chunk_v + 1);
        uint32_t* d_vfmask = plan.fmask ? B.alloc<uint32_t>(chunk_v + 1) : nullptr;
        uint32_t* d_voff = nullptr; size_t voff_cap = 0;
        MatchArena chunk{B.alloc<MatchRec>(plan.chunk_match_cap), plan.chunk_match_cap, "more than 2^31 matches in one chunk; lower GSX_VARIANT_CHUNK"};
        d_matches = B.alloc<MatchRec>(match_cap);
        CK(cudaMemsetAsync(d_ctrs, 0, 8 * sizeof(uint32_t), s));
        CK(cudaMemsetAsync(d_nmatch, 0, (size_t)(n + 1) * 4, s));
        CK(cudaMemsetAsync(d_stats, 0, 8 * sizeof(unsigned long long), s));
        CK(cudaEventRecord(js.ev[kSweepBegin], s)); CK(cudaEventRecord(js.ev[kSweepEnd], s));
        std::vector<uint32_t> seg;                                             // {first edited guide, guide, first op list} per segment
        uint32_t n_final = 0;
        uint32_t c0 = 0, f0 = 0;                                               // next guide, and how many of its op lists are done
        while (c0 < n) {
            // as many guides as fit the chunk; a guide with more edited forms than a chunk holds is cut into runs of op lists;
            // guides dropped by the threshold pass have no edited forms
            seg.clear(); uint32_t n_v = 0;
            while (c0 < n && n_v < chunk_v) {
                const uint32_t cnt = h_dropped[c0] ? 0u : dcnt[prep.recs[job.g0 + c0].qlen];
                const uint32_t take = std::min<uint32_t>(cnt - f0, chunk_v - n_v);
                if (take) { seg.push_back(n_v); seg.push_back(c0); seg.push_back(f0); n_v += take; }
                f0 += take;
                if (f0 == cnt) { c0++; f0 = 0; } else break;                   // chunk full in the middle of a guide
            }
            const uint32_t n_seg = (uint32_t)(seg.size() / 3);
            seg.push_back(n_v);
            job.ctr.edited_guides += n_v;
            if (!n_v) continue;
            if (voff_cap < seg.size()) { if (d_voff) B.free_one(d_voff); voff_cap = std::max<size_t>(seg.size(), 4096); d_voff = B.alloc<uint32_t>(voff_cap); }
            CK(cudaMemcpyAsync(d_voff, seg.data(), seg.size() * 4, cudaMemcpyHostToDevice, s));
            LAUNCH(launch_variant_expand(d_guides, n_seg, n_v, d_voff, d_descs, d_doff, d_vq, d_vdesc, d_vguide, d_vfmask, s));
            const uint32_t sb = plan.sweep_sb(n_v, plan.edited_qmin, p.mismatches);
            if (sb) use_sweep = true;
            uint32_t h[4];
            search_until_fits(plan.search_warps, 6, spill_cap, &chunk, h, [&](uint32_t* d_spill) {
                CK(cudaMemsetAsync(d_ctrs, 0, 5 * sizeof(uint32_t), s));       // ([5], the final arena's count, stays)
                SearchArgs m = a; m.p.M = p.mismatches; m.p.R = m.p.D = 0; m.p.counting = 0; m.p.n_tasks = 2 * n_v;
                m.p.match_cap = (uint32_t)chunk.cap; m.p.spill_cap = spill_cap; m.spill = d_spill; m.matches = chunk.p;
                m.skip = nullptr; m.gq = d_vq; m.guide_nmatch = d_vnmatch; m.guides = nullptr; m.fmask = d_vfmask;
                run_fast_all_pams(m, n_v, sb, nullptr);
            });
            n_seeds += sb ? h[3] : 0;
            // room for every match of the chunk in the final arena, then rewrite (cannot overflow any more)
            if ((uint64_t)n_final + h[1] > match_cap) {
                const uint64_t cap2 = std::max<uint64_t>(match_cap * 2, ((uint64_t)n_final + h[1]) * 2);
                if (cap2 > (1ull << 31)) throw std::runtime_error("more than 2^31 matches in one batch; lower the batch size");
                MatchRec* bigger = B.alloc<MatchRec>(cap2);
                CK(cudaMemcpyAsync(bigger, d_matches, (size_t)n_final * sizeof(MatchRec), cudaMemcpyDeviceToDevice, s));
                CK(cudaStreamSynchronize(s));
                B.free_one(d_matches); d_matches = bigger; match_cap = cap2;
            }
            LAUNCH(launch_variant_rewrite(chunk.p, h[1], d_guides, d_vdesc, d_vguide, d_matches, (uint32_t)match_cap, d_ctrs + 5, d_nmatch, d_ctrs + 2, s));
            read_ctrs(&n_final, 1, d_ctrs + 5); n_launches++;
        }
        n_matches = n_final;
    }
    // every PAM of the batch over the guides of m: in one fused pass, or one pass per PAM over the same arenas (only the work
    // counters start over)
    void run_fast_all_pams(SearchArgs& m, uint32_t ng, uint32_t sb, cudaEvent_t ev_mid) {
        m.n_fused = 0;
        if (plan.fuse_pams && !m.p.counting) {
            m.n_fused = prep.n_fast_pams;
            for (uint32_t k = 0; k < prep.n_fast_pams; k++) { m.fused_pams[k] = prep.pampacks[k]; m.fused_masks[k] = prep.pammasks[k]; }
            m.plen = prep.plens[0]; m.pampack = fused_filter_pampack(prep.pampacks, prep.n_fast_pams, prep.plens[0], prep.pammasks, &m.pammask);
            launch_fast(m, ng, sb, ev_mid);
            return;
        }
        for (uint32_t k = 0; k < prep.n_fast_pams; k++) {
            m.pampack = prep.pampacks[k]; m.pammask = prep.pammasks[k]; m.plen = prep.plens[k];
            if (k) { CK(cudaMemsetAsync(d_ctrs, 0, 4, s)); CK(cudaMemsetAsync(d_ctrs + 3, 0, 8, s)); }      // task / seed-queue / work-unit counters
            launch_fast(m, ng, sb, k == 0 ? ev_mid : nullptr);
        }
    }
    // fast path launch over ng guides (m.gq): [sweep ->] search_fast_kernel [-> the two-part sweep's PAM-first search].
    // d_ctrs: [3] seed queue count, [4] sweep work-unit counter
    void launch_fast(SearchArgs& m, uint32_t ng, uint32_t sb, cudaEvent_t ev_mid) {
        const bool split = sb && plan.split;                               // (never a counting pass or edited guides: plan_search)
        if (split) sweep_split(m, ng); else if (sb) sweep_plain(m, ng, sb);
        if (sb) { m.seeds = sw.queue; m.n_seeds = d_ctrs + 3; m.seed_cap = (uint32_t)sw.queue_cap; m.combos = nullptr; m.n_combos = 0; }
        if (ev_mid) CK(cudaEventRecord(ev_mid, s));
        LAUNCH(launch_search_fast(m, plan.variant_fast, di.sm_count, s));
        if (split) finish_split(m);
    }
    // the sweep's arguments for the ng guides of m: its seed queue, gtab_rows rows of per-guide filter masks
    SweepArgs sweep_args(const SearchArgs& m, uint32_t ng, size_t gtab_rows) {
        if (!sw.queue) sw.queue = B.alloc<SeedNode>(sw.queue_cap);
        if (sw.gtab_cap < gtab_rows) { if (sw.gtab) B.free_one(sw.gtab); sw.gtab = B.alloc<uint32_t>(gtab_rows * 20); sw.gtab_cap = gtab_rows; }
        SweepArgs w{};
        w.st[0] = m.st[0]; w.st[1] = m.st[1]; w.gq = m.gq; w.skip = m.skip; w.n_guides = ng; w.M = m.p.M; w.plen = m.plen; w.pampack = m.pampack;
        w.queue = sw.queue; w.queue_cap = (uint32_t)sw.queue_cap; w.queue_count = d_ctrs + 3; w.item_counter = d_ctrs + 4;
        w.error_flag = d_ctrs + 2; w.stats = d_stats; w.gtab = sw.gtab;
        return w;
    }
    void sweep_plain(const SearchArgs& m, uint32_t ng, uint32_t sb) {
        if (sw.xtab_M != m.p.M || sw.xtab_sb != sb) {
            std::vector<uint32_t> xtab;
            sweep_make_plan(plan.ftab_L, sb, m.p.M, sw.plan, xtab);
            if (sw.xtab) B.free_one(sw.xtab);
            sw.n_xtab = (uint32_t)xtab.size(); sw.xtab_M = m.p.M; sw.xtab_sb = sb;
            xtab.resize(xtab.size() + 64, 0u);                                // (sweep_lean_kernel reads up to 63 words past a pass's end, unused)
            sw.xtab = B.alloc<uint32_t>(xtab.size());
            CK(cudaMemcpyAsync(sw.xtab, xtab.data(), xtab.size() * 4, cudaMemcpyHostToDevice, s)); CK(cudaStreamSynchronize(s));
        }
        SweepArgs w = sweep_args(m, ng, ng);
        w.plan = sw.plan; w.xtab = sw.xtab; w.n_xtab = sw.n_xtab; w.load_mode = plan.load_mode; w.fmask = m.fmask;
        w.parts = 1;                                                       // measured: cutting the units does not pay (profiles/r01r_*)
        LAUNCH(launch_sweep_guides(w, s));
        LAUNCH(launch_sweep(w, plan.sweep_variant(m.p.M, qmin, qmax, m.plen, m.pampack), di.sm_count, s));
    }
    // the two-part sweep: the distal-first form (filter-mask rows 0 .. ng-1) and the PAM-first form (rows ng .. 2ng-1) in one
    // sweep, each into its own seed queue
    void sweep_split(const SearchArgs& m, uint32_t ng) {
        if (!sp.xtab) {
            std::vector<uint32_t> xtab;
            split_make_plan(plan.ftab_L, plan.split_sb, m.p.M, 2 * kSplitHalf, prep.plen, prep.pampack, kSplitHalf, sp.plan, xtab);
            if (xtab.size() > (size_t)kSplitXtabShared) throw std::runtime_error("two-part enumeration: xor table too long for this slice width");
            sp.n_xtab = (uint32_t)xtab.size();
            sp.xtab = B.alloc<uint32_t>(xtab.size());
            CK(cudaMemcpyAsync(sp.xtab, xtab.data(), xtab.size() * 4, cudaMemcpyHostToDevice, s)); CK(cudaStreamSynchronize(s));
            sp.gq2 = B.alloc<uint64_t>(ng); sp.nmatch2 = B.alloc<uint32_t>(ng + 1);
            LAUNCH(launch_split_queries(m.gq, ng, prep.pampack, prep.plen, sp.gq2, s));
        }
        if (sp.queue2_cap != sw.queue_cap) { if (sp.queue2) B.free_one(sp.queue2); sp.queue2 = B.alloc<SeedNode>(sw.queue_cap); sp.queue2_cap = sw.queue_cap; }
        if (sp.matches2_cap < m.p.match_cap) { if (sp.matches2) B.free_one(sp.matches2); sp.matches2 = B.alloc<MatchRec>(m.p.match_cap); sp.matches2_cap = m.p.match_cap; }
        CK(cudaMemsetAsync(sp.ctrs2, 0, 4 * sizeof(uint32_t), s));
        SweepArgs w = sweep_args(m, ng, 2 * (size_t)ng);
        w.plan.L = plan.ftab_L; w.plan.sb = plan.split_sb; w.plan.M = m.p.M; w.split = sp.plan; w.gq2 = sp.gq2; w.xtab = sp.xtab; w.n_xtab = sp.n_xtab;
        w.queue2 = sp.queue2; w.queue2_count = sp.ctrs2 + 0;
        LAUNCH(launch_sweep_guides(w, s));                                 // rows 0 .. ng-1: form 0
        SweepArgs w1 = w; w1.gq = sp.gq2; w1.plen = 0; w1.pampack = 0; w1.gtab = sw.gtab + (size_t)ng * 20;
        LAUNCH(launch_sweep_guides(w1, s));                                // rows ng .. 2ng-1: form 1
        LAUNCH(launch_sweep_split(w, plan.split_ctas, di.sm_count, s));
    }
    // form 1 after form 0's tree search: the tree search of its seeds with the PAM-first query (all of it protospacer), into an
    // arena of its own, then the re-anchoring of those matches into m's arena
    void finish_split(const SearchArgs& m) {
        SearchArgs m1 = m;
        m1.gq = sp.gq2; m1.plen = 0; m1.pampack = 0; m1.seeds = sp.queue2; m1.n_seeds = sp.ctrs2 + 0;
        m1.task_counter = sp.ctrs2 + 1; m1.match_count = sp.ctrs2 + 2; m1.matches = sp.matches2; m1.guide_nmatch = sp.nmatch2;
        LAUNCH(launch_search_fast(m1, plan.variant_fast, di.sm_count, s));
        ReanchorArgs r{};
        r.st[0] = m.st[0]; r.st[1] = m.st[1]; r.in = sp.matches2; r.n_in = sp.ctrs2 + 2; r.in_cap = m.p.match_cap;
        r.gq = m.gq; r.gq2 = sp.gq2; r.pampack = prep.pampack; r.plen = prep.plen;
        r.out = m.matches; r.out_count = m.match_count; r.out_cap = m.p.match_cap; r.guide_nmatch = m.guide_nmatch; r.error_flag = m.error_flag;
        r.stats = d_stats;
        LAUNCH(launch_reanchor(r, s));
        sp.ran = true;
    }
    // matches -> per-guide hit lists in the reference's order
    void arrange() {
        HostArrays& H = job.out;
        d_moff = B.alloc<uint32_t>(n + 1);
        uint32_t* d_cursor = B.alloc<uint32_t>(n, true, s);
        uint32_t* d_by_guide = B.alloc<uint32_t>(n_matches);
        d_sorted = B.alloc<uint32_t>(n_matches);
        d_sorted_off = B.alloc<uint32_t>(n_matches);
        d_nhits = B.alloc<uint32_t>(n + 1, true, s);
        d_hoff = B.alloc<uint32_t>(n + 1);
        d_cbd = B.alloc<uint32_t>((size_t)n * n_dist, true, s);
        CK(launch_scan(d_nmatch, d_moff, n, s)); n_launches += 2 + (n_matches ? 1 : 0);
        // thousands of matches per guide (bulges): global radix sort (gsx_arrange.cu); otherwise the per-guide rank sort
        // ... and whenever SOME guide has thousands (repeat families, low-complexity guides: the rank sort is quadratic per guide -- 457 ms
        // per 200 k guides on the skew stressor of SURVEY 8(d), profiles/r02d_session_3100mb_files_cfg4_skew.jsonl)
        uint64_t max_per_guide = 0;
        if (n_matches && (uint64_t)n_matches <= (uint64_t)n * 256 && plan.order_probe) {
            unsigned long long* d_tm = B.alloc<unsigned long long>(3, true, s);
            LAUNCH(launch_total_u32(d_nmatch, n, d_tm, reinterpret_cast<unsigned int*>(d_tm + 2), reinterpret_cast<unsigned long long*>(mbox.p + 32), s));
            CK(cudaStreamSynchronize(s));
            max_per_guide = reinterpret_cast<volatile unsigned long long*>(mbox.p + 32)[1];
        }
        const int order_mode = plan.order_mode != kUnset ? plan.order_mode : (((uint64_t)n_matches > (uint64_t)n * 256 || max_per_guide > 2048) ? 2 : 0);
        if (order_mode == 2) {
            const size_t sb_bytes = order_sorted_scratch_bytes(n_matches);
            void* scratch = B.alloc<unsigned char>(sb_bytes);
            CK(launch_order_sorted(d_matches, n_matches, d_moff, n, n_dist, d_sorted, d_sorted_off, d_nhits, d_cbd, scratch, sb_bytes, s));
            n_launches += 30;                                                     // keys, radix passes, flags, scan, offsets, counts
        } else {
            CK(launch_scatter(d_matches, n_matches, d_moff, d_cursor, d_by_guide, s));
            CK(launch_order(d_matches, d_moff, d_by_guide, n, n_dist, d_sorted, d_sorted_off, d_nhits, d_cbd, order_mode == 1, s));
        }
        {   // total hits can exceed 2^32 only for absurd inputs; the scan is 32-bit, so the total is a 64-bit sum (device-side, stored
            // into the mailbox: the per-guide counts themselves travel with the other result arrays at the end)
            unsigned long long* d_tot = B.alloc<unsigned long long>(3, true, s);
            LAUNCH(launch_total_u32(d_nhits, n, d_tot, reinterpret_cast<unsigned int*>(d_tot + 2), reinterpret_cast<unsigned long long*>(mbox.p + 32), s));
            CK(cudaStreamSynchronize(s));
            const uint64_t tot = *reinterpret_cast<volatile unsigned long long*>(mbox.p + 32);
            if (tot >= (1ull << 32)) throw std::runtime_error("more than 2^32 hits in one batch; lower the batch size");
            H.n_hits = (size_t)tot;
        }
        CK(launch_scan(d_nhits, d_hoff, n, s));
        nh = (uint32_t)H.n_hits;
        d_hit_match = B.alloc<uint32_t>(nh); d_hit_row = B.alloc<uint32_t>(nh); uint32_t* d_hit_guide = B.alloc<uint32_t>(nh);
        n_launches += (n_matches ? 1 : 0) + (H.n_hits ? 1 : 0) + 2;      // scan, expand, locate_score, specificity
        CK(launch_expand(d_matches, d_moff, d_sorted, d_sorted_off, d_hoff, n, n_matches, d_hit_match, d_hit_row, d_hit_guide, s));
        CK(cudaEventRecord(js.ev[kArrangeEnd], s));
    }
    // coordinates, strands, distances and CFD of every hit
    void locate_score() {
        CK(cudaStreamWaitEvent(s, js.ev_guides, 0));                                  // the guide records (uploaded under the search)
        L.st[0] = di.st[0].d; L.st[1] = di.st[1].d; L.matches = d_matches; L.guides = d_guides; L.pamsets = d_pamsets; L.chroms = di.chroms;
        L.hit_match = d_hit_match; L.hit_row = d_hit_row; L.n_hits = nh; L.n_chr = (uint32_t)job.ix->chroms.size(); L.wide = prep.wide;
        L.genome_length = job.ix->host.genome_length;
        L.abs_pos = B.alloc<int64_t>(nh); L.chr = B.alloc<int32_t>(nh); L.pos1 = B.alloc<uint32_t>(nh); L.strand = B.alloc<uint8_t>(nh);
        L.distance = B.alloc<uint8_t>(nh); L.dna = B.alloc<uint8_t>(nh); L.rna = B.alloc<uint8_t>(nh); L.index_id = B.alloc<uint8_t>(nh);
        L.cfd = B.alloc<float>(nh); L.flags = B.alloc<uint8_t>(nh); L.stats = d_stats;
        L.key_lo = B.alloc<uint64_t>(nh); L.key_hi = prep.wide ? B.alloc<uint64_t>(nh) : nullptr; L.mlen = B.alloc<uint8_t>(nh);
        CK(launch_locate_score(L, s));
        CK(cudaEventRecord(js.ev[kLocateEnd], s));
    }
    void specificity() {
        S.guide_hoff = d_hoff; S.count_by_distance = d_cbd; S.chr = L.chr; S.cfd = L.cfd; S.flags = L.flags;
        S.counted = B.alloc<uint8_t>(nh, true, s); S.specificity = B.alloc<float>(n); S.perfect = B.alloc<uint8_t>(n);
        S.n_guides = n; S.n_dist = n_dist; S.sam_rule = p.sam_scoring ? 1 : 0; S.max_off_targets = p.max_off_targets;
        S.warp_per_guide = plan.spec_warp != kUnset ? (uint32_t)plan.spec_warp : ((uint64_t)nh > (uint64_t)n * 64 ? 1u : 0u);
        CK(launch_specificity(S, s));
        CK(cudaEventRecord(js.ev[kScoreEnd], s));
    }
    // the per-guide arrays and the per-hit arrays the caller reads (all of them for the public calls); the device's turn ends here
    void copy_results() {
        HostArrays& H = job.out;
        auto d2h = [&](void* dst, const void* src, size_t bytes) { if (bytes) CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, s)); };
        d2h(H.dropped, d_dropped, n); d2h(H.hoff, d_hoff, (size_t)(n + 1) * 4); d2h(H.n_hits_of, d_nhits, (size_t)n * 4); d2h(H.specificity, S.specificity, (size_t)n * 4);
        d2h(H.perfect, S.perfect, n); d2h(H.cbd, d_cbd, (size_t)n * n_dist * 4);
        auto hit_array = [&](uint32_t bit, auto*& dst, const auto* src) {
            using T = std::remove_pointer_t<std::remove_reference_t<decltype(dst)>>;
            if (!(job.want & bit)) { dst = nullptr; return; }
            dst = H.alloc<T>(nh); d2h(dst, src, (size_t)nh * sizeof(T));
        };
        hit_array(kWantAbsPos, H.abs_pos, L.abs_pos); hit_array(kWantSaRow, H.sa_row, d_hit_row); hit_array(kWantChr, H.chr, L.chr);
        hit_array(kWantPos1, H.pos1, L.pos1); hit_array(kWantStrand, H.strand, L.strand); hit_array(kWantDistance, H.distance, L.distance);
        hit_array(kWantBulges, H.rna, L.rna); hit_array(kWantBulges, H.dna, L.dna); hit_array(kWantIndexId, H.index_id, L.index_id);
        hit_array(kWantCfd, H.cfd, L.cfd); hit_array(kWantCounted, H.counted, S.counted);
        hit_array(kWantMatchString, H.key_lo, L.key_lo); hit_array(kWantMatchString, H.mlen, L.mlen);
        H.key_hi = nullptr; if (prep.wide) hit_array(kWantMatchString, H.key_hi, L.key_hi);
        d2h(stats, d_stats, sizeof stats);
        CK(cudaEventRecord(js.ev[kCopyEnd], s));
        CK(cudaStreamSynchronize(s)); CK(cudaStreamSynchronize(s2));
        // the turn on the device ends with the copies: a result transfer running under the NEXT call's sweep slows both several
        // times over (170 MB streaming through the L2 that holds the sweep's slices: profiles/r02b_session_3100mb_sweep_lean.jsonl,
        // m3_lean_v11_pipe2); what overlaps between pipelined calls is the host work -- guide packing before, result assembly after
        if (turn.owns_lock()) turn.unlock();
    }
    void counters() {
        gsx_counters& c = job.ctr;
        auto ms = [&](JobEvent a0, JobEvent a1) { float t; CK(cudaEventElapsedTime(&t, js.ev[a0], js.ev[a1])); return (double)t; };
        c.ms_search = ms(kSearchBegin, kSearchEnd); c.ms_arrange = ms(kSearchEnd, kArrangeEnd); c.ms_locate = ms(kArrangeEnd, kLocateEnd);
        c.ms_score = ms(kLocateEnd, kScoreEnd); c.ms_total_device = ms(kSearchBegin, kScoreEnd); c.ms_d2h = ms(kScoreEnd, kCopyEnd);
        c.ms_sweep = ms(kSweepBegin, kSweepEnd); c.seeds = n_seeds;
        c.sectors = use_sweep ? stats[5] + stats[7] : stats[1];
        c.nodes = stats[0]; c.lookups = stats[1]; c.spills = stats[2]; c.lf_steps = stats[3];
        c.matches = n_matches; c.hits = nh; c.launches = n_launches;
    }
};


static void run_device_job(DeviceJob* job) {
    try {
        CK(cudaSetDevice(job->ix->dev[job->slot].device));
        DeviceRun r(*job);
        if (!r.setup()) return;
        if (job->p->threshold > 0) r.threshold_pass();
        r.search();
        r.arrange();
        r.locate_score();
        r.specificity();
        r.copy_results();
        r.counters();
    } catch (const CudaError& e) { job->status = GSX_ERR_CUDA; job->err = e.what(); }
    catch (const std::bad_alloc&) { job->status = GSX_ERR_NOMEM; job->err = "out of host memory"; }
    catch (const std::exception& e) { job->status = GSX_ERR_INTERNAL; job->err = e.what(); }
}
#undef LAUNCH

// The public view.  One part: its arrays as they are.  Several parts (one per device): the per-guide and per-hit arrays are
// concatenated -- lazily, when gsx_result_view_get is first called; the library's own formatter reads the parts in place.
static void merge_parts(gsx_result* r) {
    gsx_result_view& v = r->view;
    auto cat = [&](auto& dst, auto member, bool per_hit, size_t mult) {
        dst.clear();
        for (auto& p : r->parts) { size_t n = (per_hit ? p.n_hits : p.n_guides) * mult; auto* src = p.*member; if (n && src) dst.insert(dst.end(), src, src + n); }
    };
    cat(r->dropped, &HostArrays::dropped, false, 1); cat(r->n_hits_of, &HostArrays::n_hits_of, false, 1);
    cat(r->specificity, &HostArrays::specificity, false, 1); cat(r->perfect, &HostArrays::perfect, false, 1);
    cat(r->cbd, &HostArrays::cbd, false, r->n_dist);
    cat(r->abs_pos, &HostArrays::abs_pos, true, 1); cat(r->sa_row, &HostArrays::sa_row, true, 1); cat(r->chr, &HostArrays::chr, true, 1);
    cat(r->pos1, &HostArrays::pos1, true, 1); cat(r->strand, &HostArrays::strand, true, 1); cat(r->distance, &HostArrays::distance, true, 1);
    cat(r->rna, &HostArrays::rna, true, 1); cat(r->dna, &HostArrays::dna, true, 1); cat(r->index_id, &HostArrays::index_id, true, 1);
    cat(r->cfd, &HostArrays::cfd, true, 1); cat(r->counted, &HostArrays::counted, true, 1);
    v.dropped = r->dropped.data(); v.n_hits_of = r->n_hits_of.data(); v.specificity = r->specificity.data(); v.perfect_match = r->perfect.data();
    v.count_by_distance = r->cbd.data(); v.abs_pos = r->abs_pos.data(); v.sa_row = r->sa_row.data(); v.chr = r->chr.data(); v.pos1 = r->pos1.data();
    v.strand = r->strand.data(); v.distance = r->distance.data(); v.rna_bulges = r->rna.data(); v.dna_bulges = r->dna.data();
    v.index_id = r->index_id.data(); v.cfd = r->cfd.data(); v.counted = r->counted.data();
}

void gsx_build_view(gsx_result* r) {
    gsx_result_view& v = r->view;
    size_t ng = 0, nh = 0;
    for (auto& p : r->parts) { ng += p.n_guides; nh += p.n_hits; }
    v.n_guides = ng; v.n_hits = nh; v.n_dist = r->n_dist;
    r->first_hit.resize(ng + 1);                                             // (one entry more than guides: the end of the last guide's hits)
    size_t g = 0, h = 0;
    for (auto& p : r->parts) { for (size_t i = 0; i < p.n_guides; i++) r->first_hit[g + i] = h + p.hoff[i]; g += p.n_guides; h += p.n_hits; }
    r->first_hit[ng] = nh;
    v.first_hit = r->first_hit.data();
    r->merged = r->parts.size() == 1;
    if (r->parts.size() == 1) {
        HostArrays& p = r->parts[0];
        v.dropped = p.dropped; v.n_hits_of = p.n_hits_of; v.specificity = p.specificity; v.perfect_match = p.perfect; v.count_by_distance = p.cbd;
        v.abs_pos = p.abs_pos; v.sa_row = p.sa_row; v.chr = p.chr; v.pos1 = p.pos1; v.strand = p.strand; v.distance = p.distance;
        v.rna_bulges = p.rna; v.dna_bulges = p.dna; v.index_id = p.index_id; v.cfd = p.cfd; v.counted = p.counted;
    }
}

static int enumerate_impl(const gsx_index* ix, const gsx_guide* guides, size_t n_guides, const gsx_params* p, gsx_result** out, uint32_t want);
extern "C" int gsx_enumerate(const gsx_index* ix, const gsx_guide* guides, size_t n_guides, const gsx_params* p, gsx_result** out) {
    if (!ix || !p || !out || (!guides && n_guides)) return fail(GSX_ERR_ARG, "null argument");
    *out = nullptr;
    return guarded([&] { return enumerate_impl(ix, guides, n_guides, p, out, kWantAll); });
}
static int enumerate_impl(const gsx_index* ix, const gsx_guide* guides, size_t n_guides, const gsx_params* p, gsx_result** out, uint32_t want) {
    if (ix->dev.empty()) return fail(GSX_ERR_NO_DEVICE, "index is not resident on any device");
    if (n_guides >= (1ull << 30)) return fail(GSX_ERR_ARG, "too many guides in one call");
    const auto t_call = std::chrono::steady_clock::now();
    Prepared prep;
    if (int rc = gsx_prepare_guides(guides, n_guides, p, prep)) return rc;
    const double ms_prepare = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_call).count();
    const size_t nd = ix->dev.size();
    // guides are independent: contiguous shards per device, no data-path collective (SURVEY.md 8(e))
    std::vector<DeviceJob> jobs(nd);
    for (size_t d = 0; d < nd; d++) {
        jobs[d].ix = ix; jobs[d].slot = (int)d; jobs[d].prep = &prep; jobs[d].p = p; jobs[d].want = want;
        jobs[d].g0 = n_guides * d / nd; jobs[d].g1 = n_guides * (d + 1) / nd;
    }
    if (nd == 1) run_device_job(&jobs[0]);
    else { std::vector<std::thread> th; for (auto& j : jobs) th.emplace_back(run_device_job, &j); for (auto& t : th) t.join(); }
    for (auto& j : jobs) if (j.status != GSX_OK) { for (auto& k : jobs) k.out.release(); return fail(j.status, j.err); }
    gsx_result* r = new gsx_result();
    r->n_dist = p->mismatches + 1; r->wide = prep.wide; r->guides = std::move(prep.recs);
    size_t g = 0, h = 0;
    for (auto& j : jobs) {
        r->part_g0.push_back(g); r->part_h0.push_back(h); g += j.out.n_guides; h += j.out.n_hits;
        r->parts.push_back(std::move(j.out));
        gsx_counters& c = r->counters;
        c.nodes += j.ctr.nodes; c.lookups += j.ctr.lookups; c.matches += j.ctr.matches; c.hits += j.ctr.hits; c.lf_steps += j.ctr.lf_steps; c.spills += j.ctr.spills; c.launches += j.ctr.launches; c.seeds += j.ctr.seeds; c.sectors += j.ctr.sectors; c.edited_guides += j.ctr.edited_guides;
        c.ms_sweep = std::max(c.ms_sweep, j.ctr.ms_sweep);
        c.ms_search = std::max(c.ms_search, j.ctr.ms_search); c.ms_arrange = std::max(c.ms_arrange, j.ctr.ms_arrange);
        c.ms_locate = std::max(c.ms_locate, j.ctr.ms_locate); c.ms_score = std::max(c.ms_score, j.ctr.ms_score);
        c.ms_total_device = std::max(c.ms_total_device, j.ctr.ms_total_device); c.ms_h2d = std::max(c.ms_h2d, j.ctr.ms_h2d); c.ms_d2h = std::max(c.ms_d2h, j.ctr.ms_d2h);
    }
    gsx_build_view(r);
    r->counters.ms_prepare = ms_prepare;
    r->counters.ms_wall = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_call).count();
    *out = r;
    return GSX_OK;
}

// ---- two-slot form: the call runs on a library thread, the caller prepares / consumes another batch meanwhile ----------------
struct gsx_pending {
    std::thread th; gsx_result* result = nullptr; int status = GSX_OK; std::string err;
};
extern "C" int gsx_enumerate_start(const gsx_index* ix, const gsx_guide* guides, size_t n_guides, const gsx_params* p, gsx_pending** out) {
    return gsx_internal_enumerate_start_want(ix, guides, n_guides, p, kWantAll, out);
}
// (not in include/gsx.h: the whole-file driver's form of the call, bringing only the per-hit arrays it formats from -- gsx_host.h)
extern "C" int gsx_internal_enumerate_start_want(const gsx_index* ix, const gsx_guide* guides, size_t n_guides, const gsx_params* p, uint32_t want, gsx_pending** out) {
    if (!ix || !p || !out || (!guides && n_guides)) return fail(GSX_ERR_ARG, "null argument");
    *out = nullptr;
    return guarded([&] {
        gsx_pending* pd = new gsx_pending();
        try {
            pd->th = std::thread([=] {
                pd->result = nullptr;
                pd->status = guarded([&] { return enumerate_impl(ix, guides, n_guides, p, &pd->result, want); });
                if (pd->status) pd->err = g_err;                            // (the message lives in the worker thread's slot)
            });
        } catch (...) { delete pd; throw; }
        *out = pd;
        return (int)GSX_OK;
    });
}
extern "C" int gsx_enumerate_wait(gsx_pending* pd, gsx_result** out) {
    if (!pd || !out) return fail(GSX_ERR_ARG, "null argument");
    if (pd->th.joinable()) pd->th.join();
    *out = pd->result;
    const int rc = pd->status; const std::string msg = pd->err;
    delete pd;
    return rc ? fail(rc, msg) : (int)GSX_OK;
}

extern "C" int gsx_result_view_get(const gsx_result* r, gsx_result_view* view) {
    if (!r || !view) return fail(GSX_ERR_ARG, "null argument");
    return guarded([&] {
        gsx_result* w = const_cast<gsx_result*>(r);                             // (the merged copy is a cache: built once, under the result's own lock)
        std::lock_guard<std::mutex> lk(w->merge_mu);
        if (!w->merged) { merge_parts(w); w->merged = true; }
        *view = w->view;
        return (int)GSX_OK;
    });
}
extern "C" int gsx_result_counters(const gsx_result* r, gsx_counters* out) { if (!r || !out) return fail(GSX_ERR_ARG, "null argument"); *out = r->counters; return GSX_OK; }

extern "C" int gsx_result_match_sequence(const gsx_result* r, size_t hit, char* buf, size_t buf_len) {
    if (!r || !buf || buf_len < 48) return fail(GSX_ERR_ARG, "buffer must hold 48 bytes");
    if (hit >= r->view.n_hits) return fail(GSX_ERR_ARG, "hit index out of range");
    size_t pi = std::upper_bound(r->part_h0.begin(), r->part_h0.end(), hit) - r->part_h0.begin() - 1;
    const HostArrays& p = r->parts[pi];
    const size_t hl = hit - r->part_h0[pi];
    MatchRec m{}; m.key_lo = p.key_lo[hl]; m.key_hi = p.key_hi ? p.key_hi[hl] : 0; m.info = (uint32_t)p.mlen[hl] << 24;
    // the guide of the hit: the last one whose first hit is not behind it (guides without hits share their successor's offset)
    const size_t gi = (size_t)(std::upper_bound(r->first_hit.begin(), r->first_hit.end() - 1, (uint64_t)hit) - r->first_hit.begin()) - 1;
    const GuideRec& g = r->guides[gi];
    uint32_t len = decode_match(m, g, r->wide, buf);
    for (uint32_t i = 0; i < len; i++) buf[i] = complement_char(buf[i]);
    buf[len] = 0;
    return GSX_OK;
}

extern "C" void gsx_result_free(gsx_result* r) {
    if (!r) return;
    for (auto& p : r->parts) p.release();
    {
        std::lock_guard<std::mutex> lk(g_recs_mu);
        if (g_recs_free.size() < 4 && r->guides.capacity()) g_recs_free.push_back(std::move(r->guides));
    }
    delete r;
}

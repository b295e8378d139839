// guidescan -- host CLI with the reference's `index` / `enumerate` command line (reference src/guidescan.cxx:28-95,
// 316-358; option spellings and defaults: SURVEY.md section 8(b)), driving the GPU path through the C ABI.
// Text formatting, file I/O and option parsing are host C++; all arithmetic of the hot path runs on the device.
#include "../../include/gsx.h"
#include <algorithm>
#include <cerrno>
#include <chrono>
#include <fcntl.h>
#include <sys/stat.h>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

static void usage() {
    fprintf(stderr,
            "Guidescan all-in-one interface (B200 build).\n"
            "Usage: guidescan [--version] SUBCOMMAND ...\n\n"
            "  index [--index PREFIX] [--reference-format] GENOME.fa\n"
            "      Builds a genomic index over a FASTA file (GPU suffix sorting; writes PREFIX.gsx + PREFIX.gs).\n"
            "      --reference-format          Also write PREFIX.forward / PREFIX.reverse, the files of the original guidescan (extension).\n"
            "  enumerate [OPTIONS] INDEX_PREFIX\n"
            "      --start                     Match PAM at start of kmer instead at end (default).\n"
            "      --max-off-targets INT=-1    Maximum number of off-targets to store for each number of mismatches.\n"
            "      -n,--threads UINT           Host worker threads that format the output (default: all cores); the search runs on the GPU(s).\n"
            "      -a,--alt-pam TEXT ...       Alternative PAMs used to find off-targets\n"
            "      --iupac-pam                 Read the kmers file's PAM column and -a with IUPAC class letters (R, Y, S, W, K, M,\n"
            "                                  B, D, H, V: a class matches its member bases, never a genome N); without it any\n"
            "                                  letter but A, C, G, T, N never matches (extension; set by itself for a --pam with one).\n"
            "      -m,--mismatches UINT=3      Number of mismatches to allow when finding off-targets\n"
            "      --rna-bulges UINT=0         Max number of RNA bulges to allow when finding off-targets\n"
            "      --dna-bulges UINT=0         Number of DNA bulges to allow when finding off-targets\n"
            "      -t,--threshold INT=-1       Filters gRNAs with off-targets at a distance at or below this threshold\n"
            "      --format TEXT:{csv,sam}     File format for output.\n"
            "      --mode TEXT:{succinct,complete}  Information to output.\n"
            "      -f,--kmers-file FILE        REQUIRED  File containing kmers to build gRNA database over\n"
            "                                  (unless --genome is given; the two are mutually exclusive)\n"
            "      -o,--output TEXT            REQUIRED  Output file.\n"
            "      --gpus INT=1                Number of GPUs to shard the guides over (extension): devices 0 .. INT-1.\n"
            "      --devices LIST              The same with explicit device ordinals, e.g. 0,2,3 (extension).\n"
            "      --genome GENOME.fa          Generate the guides from this FASTA (as `kmers` does, PAM position from --start) and\n"
            "                                  enumerate them in one pass, without a kmers file (extension).  With --genome:\n"
            "        --pam TEXT=NGG            PAM pattern (A, C, G, T, N and IUPAC class letters, e.g. NRG, NNGRRT, TTTV).\n"
            "        --kmer-length UINT=20     Guide length, 1..32 (with the PAM and DNA bulges at most 32).\n"
            "        --min-chr-length UINT=0   Skip FASTA records shorter than this.\n"
            "        --prefix TEXT             Prefix of every guide id.\n"
            "        --regions BED             Keep only guides whose k bases lie inside one BED interval (0-based, half-open).\n"
            "  kmers [OPTIONS] GENOME.fa\n"
            "      Writes the kmers file `enumerate -f` reads: every k-mer next to a PAM on either strand (the original's\n"
            "      scripts/generate_kmers.py; the PAM scan runs on the GPU).\n"
            "      -o,--output FILE            REQUIRED  Output CSV.\n"
            "      --pam TEXT=NGG              PAM pattern (A, C, G, T, N and IUPAC class letters, expanded like N).\n"
            "      --kmer-length UINT=20       Length of the k-mers.\n"
            "      --min-chr-length UINT=0     Skip FASTA records shorter than this.\n"
            "      --prefix TEXT               Prefix of every k-mer id.\n"
            "      --start                     The PAM precedes the k-mer.\n"
            "      --device INT=0              GPU that runs the scan.\n"
            "  decode [OPTIONS] DATABASE.sam\n"
            "      Turns the of:H: off-target lists of a database written with --format sam --mode complete back into enumerate's\n"
            "      CSV rows (the original's scripts/decode_database.py; sites and CFD computed on the GPU).\n"
            "      --genome GENOME.fa          REQUIRED  The assembly the database was computed on.\n"
            "      -o,--output FILE            REQUIRED  Output CSV.\n"
            "      --mode TEXT:{succinct,complete}  Columns, as enumerate's (default complete).\n"
            "      --cfd                       Append a cfd column.\n"
            "      --pam-length UINT=3         Characters of the PAM column at the end of each sequence.\n"
            "      -a,--alt-pam TEXT ...       Alternative PAMs the database was written with (IUPAC class letters allowed).\n"
            "      --regions BED               Only guides whose on-target site lies inside one BED interval (0-based, half-open).\n"
            "      --device INT=0              GPU that decodes.\n");
}

static std::string lower(std::string s) { std::transform(s.begin(), s.end(), s.begin(), ::tolower); return s; }

// a non-negative decimal option value; anything else ends the program with the CLI's usage status
static unsigned long long uint_arg(const char* name, const char* v) {
    char* end = nullptr;
    errno = 0;
    const unsigned long long x = strtoull(v, &end, 10);
    if (!*v || *end || errno || v[0] == '-') { fprintf(stderr, "%s: %s is not a non-negative integer\n", name, v); exit(105); }
    return x;
}

// PAM characters of the generator and the decoder: A, C, G, T, N and the upper-case IUPAC class letters
static bool is_class(char c) { return c && strchr("RYSWKMBDHV", c) != nullptr; }
static bool pam_ok(const std::string& pam) {
    if (pam.empty() || pam.size() > 8) return false;
    for (char c : pam) if (!(c == 'A' || c == 'C' || c == 'G' || c == 'T' || c == 'N' || is_class(c))) return false;
    return true;
}
static const char* kPamLetters = "A, C, G, T, N or IUPAC class letters (R, Y, S, W, K, M, B, D, H, V)";

static int do_kmers(int argc, char** argv) {
    std::string fasta, output, pam = "NGG", prefix;
    unsigned long long k = 20, min_len = 0, device = 0; bool start = false;
    for (int i = 0; i < argc; i++) {
        std::string a = argv[i];
        auto need = [&](const char* name) -> const char* { if (i + 1 >= argc) { fprintf(stderr, "%s: 1 required\n", name); exit(106); } return argv[++i]; };
        if (a == "-o" || a == "--output") output = need("--output");
        else if (a == "--pam") pam = need("--pam");
        else if (a == "--kmer-length") k = uint_arg("--kmer-length", need("--kmer-length"));
        else if (a == "--min-chr-length") min_len = uint_arg("--min-chr-length", need("--min-chr-length"));
        else if (a == "--prefix") prefix = need("--prefix");
        else if (a == "--start") start = true;
        else if (a == "--device") device = uint_arg("--device", need("--device"));
        else if (a == "-h" || a == "--help") { usage(); return 0; }
        else if (!a.empty() && a[0] == '-') { fprintf(stderr, "The following argument was not expected: %s\n", a.c_str()); return 109; }
        else fasta = a;
    }
    if (fasta.empty()) { fprintf(stderr, "genome is required\n"); return 106; }
    if (output.empty()) { fprintf(stderr, "--output is required\n"); return 106; }
    if (k < 1 || k > 64) { fprintf(stderr, "--kmer-length: %llu not in 1..64\n", k); return 105; }
    if (!pam_ok(pam)) { fprintf(stderr, "--pam: %s must be 1..8 characters of %s\n", pam.c_str(), kPamLetters); return 105; }
    uint64_t n = 0;
    const auto t0 = std::chrono::steady_clock::now();
    if (gsx_generate_kmers(fasta.c_str(), output.c_str(), pam.c_str(), (uint32_t)k, min_len, prefix.c_str(), start, (int)device, &n)) {
        fprintf(stderr, "ERROR: %s\n", gsx_last_error()); return 1;
    }
    printf("Wrote %llu kmer(s) to %s in %.3f s.\n", (unsigned long long)n, output.c_str(), std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count());
    return 0;
}

static int do_decode(int argc, char** argv) {
    std::string sam, genome, output, mode = "complete", regions;
    std::vector<std::string> alts; unsigned long long pam_length = 3, device = 0; bool cfd = false;
    for (int i = 0; i < argc; i++) {
        std::string a = argv[i];
        auto need = [&](const char* name) -> const char* { if (i + 1 >= argc) { fprintf(stderr, "%s: 1 required\n", name); exit(106); } return argv[++i]; };
        if (a == "-o" || a == "--output") output = need("--output");
        else if (a == "--genome") genome = need("--genome");
        else if (a == "--mode") mode = lower(need("--mode"));
        else if (a == "--cfd") cfd = true;
        else if (a == "--pam-length") pam_length = uint_arg("--pam-length", need("--pam-length"));
        else if (a == "-a" || a == "--alt-pam") { while (i + 1 < argc && argv[i + 1][0] != '-') alts.push_back(argv[++i]); }
        else if (a == "--regions") regions = need("--regions");
        else if (a == "--device") device = uint_arg("--device", need("--device"));
        else if (a == "-h" || a == "--help") { usage(); return 0; }
        else if (!a.empty() && a[0] == '-') { fprintf(stderr, "The following argument was not expected: %s\n", a.c_str()); return 109; }
        else sam = a;
    }
    if (sam.empty()) { fprintf(stderr, "database is required\n"); return 106; }
    if (genome.empty()) { fprintf(stderr, "--genome is required\n"); return 106; }
    if (output.empty()) { fprintf(stderr, "--output is required\n"); return 106; }
    if (mode != "succinct" && mode != "complete") { fprintf(stderr, "--mode: %s not in {succinct,complete}\n", mode.c_str()); return 105; }
    if (pam_length < 1 || pam_length > 8) { fprintf(stderr, "--pam-length: %llu not in 1..8\n", pam_length); return 105; }
    for (auto& x : alts)
        if (!pam_ok(x) || x.size() != pam_length) { fprintf(stderr, "--alt-pam: %s must be %llu characters of %s\n", x.c_str(), pam_length, kPamLetters); return 105; }
    std::vector<const char*> ap; for (auto& s : alts) ap.push_back(s.c_str());
    size_t ng = 0, nr = 0;
    const auto t0 = std::chrono::steady_clock::now();
    if (gsx_decode_database(sam.c_str(), genome.c_str(), output.c_str(), (uint32_t)pam_length, ap.data(), (uint32_t)ap.size(), mode == "complete", cfd,
                            regions.empty() ? nullptr : regions.c_str(), (int)device, &ng, &nr)) {
        fprintf(stderr, "ERROR: %s\n", gsx_last_error()); return 1;
    }
    printf("Decoded %zu guide(s) into %zu row(s) in %s in %.3f s.\n", ng, nr, output.c_str(), std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count());
    return 0;
}

static int do_index(int argc, char** argv) {
    std::string fasta, prefix; bool reference_format = false;
    for (int i = 0; i < argc; i++) {
        std::string a = argv[i];
        if (a == "--index" && i + 1 < argc) prefix = argv[++i];
        else if (a == "--reference-format") reference_format = true;
        else if (a.rfind("--index=", 0) == 0) prefix = a.substr(8);
        else fasta = a;
    }
    if (fasta.empty()) { fprintf(stderr, "genome is required\n"); return 106; }
    if (prefix.empty()) { prefix = fasta + ".index"; printf("Index file prefix not specified. Using default: %s\n", prefix.c_str()); }
    gsx_index* ix = nullptr;
    int rc = gsx_index_build(fasta.c_str(), prefix.c_str(), nullptr, 0, &ix);
    if (rc) { fprintf(stderr, "ERROR: %s\n", gsx_last_error()); return 1; }
    if (reference_format) {
        const auto t0 = std::chrono::steady_clock::now();
        if (gsx_index_save_reference_format(ix, prefix.c_str())) { fprintf(stderr, "ERROR: %s\n", gsx_last_error()); gsx_index_close(ix); return 1; }
        utimensat(AT_FDCWD, (prefix + ".gsx").c_str(), nullptr, 0);     // gsx_index_open takes the newer format: keep that the one without conversion
        printf("Wrote %s.forward and %s.reverse in %.2f s.\n", prefix.c_str(), prefix.c_str(), std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count());
    }
    printf("Index construction complete.\n");
    gsx_index_close(ix);
    return 0;
}

static int do_enumerate(int argc, char** argv) {
    gsx_params p; gsx_params_default(&p);
    std::string index, kmers, output, format = "csv", mode = "complete";
    std::vector<std::string> alts; int gpus = 1; std::vector<int> devs;
    // --genome: the generator's options (`kmers`) and the regions; `generator` lists those given, which -f does not take
    std::string genome, pam = "NGG", prefix, regions; unsigned long long k = 20, min_len = 0; std::vector<std::string> generator;
    for (int i = 0; i < argc; i++) {
        std::string a = argv[i];
        auto need = [&](const char* name) -> const char* { if (i + 1 >= argc) { fprintf(stderr, "%s: 1 required\n", name); exit(106); } return argv[++i]; };
        if (a == "--start") p.start = 1;
        else if (a == "--iupac-pam") p.iupac_pams = 1;
        else if (a == "--max-off-targets") p.max_off_targets = atoll(need("--max-off-targets"));
        else if (a == "-n" || a == "--threads") { const int t = atoi(need("--threads")); if (t > 0) setenv("GSX_FORMAT_THREADS", std::to_string(t).c_str(), 1); }
        else if (a == "-a" || a == "--alt-pam") {          // greedy multi-value, as CLI11 parses it (SURVEY.md App. E.7)
            while (i + 1 < argc && argv[i + 1][0] != '-') alts.push_back(argv[++i]);
        }
        else if (a == "-m" || a == "--mismatches") p.mismatches = (uint32_t)atoi(need("--mismatches"));
        else if (a == "--rna-bulges") p.rna_bulges = (uint32_t)atoi(need("--rna-bulges"));
        else if (a == "--dna-bulges") p.dna_bulges = (uint32_t)atoi(need("--dna-bulges"));
        else if (a == "-t" || a == "--threshold") p.threshold = atoi(need("--threshold"));
        else if (a == "--format") format = lower(need("--format"));
        else if (a == "--mode") mode = lower(need("--mode"));
        else if (a == "-f" || a == "--kmers-file") kmers = need("--kmers-file");
        else if (a == "-o" || a == "--output") output = need("--output");
        else if (a == "--genome") genome = need("--genome");
        else if (a == "--pam") { pam = need("--pam"); generator.push_back(a); }
        else if (a == "--kmer-length") { k = uint_arg("--kmer-length", need("--kmer-length")); generator.push_back(a); }
        else if (a == "--min-chr-length") { min_len = uint_arg("--min-chr-length", need("--min-chr-length")); generator.push_back(a); }
        else if (a == "--prefix") { prefix = need("--prefix"); generator.push_back(a); }
        else if (a == "--regions") { regions = need("--regions"); generator.push_back(a); }
        else if (a == "--gpus") gpus = atoi(need("--gpus"));
        else if (a == "--devices") {
            std::string l = need("--devices");
            for (size_t b = 0; b < l.size();) { size_t e = l.find(',', b); if (e == std::string::npos) e = l.size(); if (e > b) devs.push_back(atoi(l.substr(b, e - b).c_str())); b = e + 1; }
        }
        else if (a == "-h" || a == "--help") { usage(); return 0; }
        else if (!a.empty() && a[0] == '-') { fprintf(stderr, "The following argument was not expected: %s\n", a.c_str()); return 109; }
        else index = a;
    }
    if (index.empty()) { fprintf(stderr, "index is required\n"); return 106; }
    if (!kmers.empty() && !genome.empty()) { fprintf(stderr, "--kmers-file excludes --genome: give one of them\n"); return 109; }
    if (kmers.empty() && genome.empty()) { fprintf(stderr, "--kmers-file is required\n"); return 106; }
    if (genome.empty() && !generator.empty()) { fprintf(stderr, "%s needs --genome\n", generator[0].c_str()); return 109; }
    if (output.empty()) { fprintf(stderr, "--output is required\n"); return 106; }
    if (format != "csv" && format != "sam") { fprintf(stderr, "--format: %s not in {csv,sam}\n", format.c_str()); return 105; }
    if (mode != "succinct" && mode != "complete") { fprintf(stderr, "--mode: %s not in {succinct,complete}\n", mode.c_str()); return 105; }
    if (!genome.empty()) {                                    // (the library checks these too; here they fail before the index is opened)
        if (k < 1 || k > 32) { fprintf(stderr, "--kmer-length: %llu not in 1..32\n", k); return 105; }
        if (!pam_ok(pam)) { fprintf(stderr, "--pam: %s must be 1..8 characters of %s\n", pam.c_str(), kPamLetters); return 105; }
        for (char c : pam) if (is_class(c)) p.iupac_pams = 1;      // the generated guides carry the pattern as their PAM column
        size_t longest = pam.size(); for (auto& x : alts) longest = std::max(longest, x.size());
        if (k + longest + p.dna_bulges > 32) { fprintf(stderr, "--kmer-length %llu + PAM %zu + --dna-bulges %u is longer than 32\n", k, longest, p.dna_bulges); return 105; }
    }
    std::vector<const char*> ap; for (auto& s : alts) ap.push_back(s.c_str());
    p.alt_pams = ap.data(); p.n_alt_pams = (uint32_t)ap.size();
    if (devs.empty()) for (int d = 0; d < std::max(1, gpus); d++) devs.push_back(d);
    printf("Loading genome index at \"%s\".\n", index.c_str());
    gsx_index* ix = nullptr;
    int rc = gsx_index_open(index.c_str(), devs.data(), (int)devs.size(), &ix);
    if (rc) { fprintf(stderr, "%s\n", gsx_last_error()); return 1; }
    {
        double t[3] = {0, 0, 0}; gsx_index_open_seconds(ix, t);
        printf("Successfully loaded genome index. (%zu device(s): files %.2f s, device layout %.2f s, replication %.2f s)\n", devs.size(), t[0], t[1], t[2]);
    }
    auto t0 = std::chrono::steady_clock::now();
    size_t n = 0; gsx_counters c;
    if (genome.empty()) rc = gsx_enumerate_file(ix, kmers.c_str(), output.c_str(), &p, format == "sam", mode == "complete", 0, &n, &c);
    else rc = gsx_enumerate_genome(ix, genome.c_str(), pam.c_str(), (uint32_t)k, min_len, prefix.c_str(), regions.empty() ? nullptr : regions.c_str(),
                                   output.c_str(), &p, format == "sam", mode == "complete", 0, &n, &c);
    if (rc) { fprintf(stderr, "%s\n", gsx_last_error()); gsx_index_close(ix); return 1; }
    double secs = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    printf("Read in %zu kmer(s).\n", n);
    printf("Processed %zu kmers in %lld seconds. (%.3f s, %.1f kmers/s; device %.1f ms; %llu nodes, %llu hits)\n", n, (long long)secs, secs,
           secs > 0 ? n / secs : 0.0, c.ms_total_device, (unsigned long long)c.nodes, (unsigned long long)c.hits);
    gsx_index_close(ix);
    return 0;
}

int main(int argc, char** argv) {
    if (argc < 2) { usage(); return 106; }
    std::string cmd = argv[1];
    if (cmd == "--version") { printf("%s\n", gsx_version()); return 0; }
    if (cmd == "-h" || cmd == "--help") { usage(); return 0; }
    if (cmd == "index") return do_index(argc - 2, argv + 2);
    if (cmd == "enumerate") return do_enumerate(argc - 2, argv + 2);
    if (cmd == "kmers") return do_kmers(argc - 2, argv + 2);
    if (cmd == "decode") return do_decode(argc - 2, argv + 2);
    if (cmd == "download") { fprintf(stderr, "download: not part of the GPU hot path (no network); use the reference binary\n"); return 1; }
    usage();
    return 106;
}

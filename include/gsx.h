/*
 * gsx.h -- C ABI of the B200-native off-target enumeration path (libgsx.so).
 *
 * The reference (pritykinlab/guidescan-cli 2.0.0) has no plugin / FFI surface: its hot path is header
 * templates inlined into one translation unit.  The seam this ABI sits behind is the set of calls that
 * `process_kmer_to_stream` makes for every guide (reference include/genomics/process.hpp:35-128):
 *
 *   genome_index::inexact_search(query, pams, mismatches, rna, dna, 1, cb, data)   include/genomics/index.hpp:102-110,377-398
 *   genome_index::resolve(bwt_position)                                            include/genomics/index.hpp:53-55
 *   resolve_absolute(gs, abs, kmer)                                                src/genomics/structures.cxx:7-52
 *   calculate_cfd / specificity reduction                                          include/genomics/printer.hpp:98-113,244-300
 *   get_csv_lines / get_sam_lines                                                  include/genomics/printer.hpp:244-360
 *
 * batched over guides (the reference handles one guide per call; a GPU wants 10^4..10^6 at once).
 * Plain C types only; no C++ exceptions cross this boundary; every function returns 0 on success or a
 * gsx_status code, with a thread-local message available from gsx_last_error().
 * There is NO CPU fallback: without a CUDA device every compute entry point fails with GSX_ERR_NO_DEVICE.
 */
#ifndef GSX_H
#define GSX_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
    GSX_OK = 0,
    GSX_ERR_ARG = 1,          /* bad argument / unsupported option range */
    GSX_ERR_IO = 2,           /* missing or malformed index / input file (reference: log line + return 1, src/guidescan.cxx:193-208) */
    GSX_ERR_NO_DEVICE = 3,    /* no usable CUDA device (there is no CPU path) */
    GSX_ERR_CUDA = 4,         /* CUDA runtime error, message carries cudaGetErrorString */
    GSX_ERR_NOMEM = 5,
    GSX_ERR_INTERNAL = 6
} gsx_status;

typedef struct gsx_index  gsx_index;     /* immutable after open; shareable across host threads (src/guidescan.cxx:198-211,243) */
typedef struct gsx_result gsx_result;

/* One candidate gRNA: the `sequence` and `pam` columns of the guides CSV (reference
 * include/genomics/structures.hpp:11-18).  NUL-terminated.  id / chromosome / position / sense stay on the host. */
typedef struct {
    const char* seq;
    const char* pam;          /* "" => the guide is searched without a PAM and alt PAMs are ignored (process.hpp:51-56) */
} gsx_guide;

/* Mirrors enumerate_cmd_options (reference include/guidescan.hpp:14-53; defaults src/guidescan.cxx:39-76). */
typedef struct {
    uint32_t mismatches;          /* -m, default 3 */
    uint32_t rna_bulges;          /* --rna-bulges, default 0 */
    uint32_t dna_bulges;          /* --dna-bulges, default 0 */
    uint32_t max_bulge_size;      /* fixed to 1 by the reference caller (process.hpp:82-87); only 1 is accepted */
    int32_t  threshold;           /* -t, default -1; active only when > 0 (process.hpp:66) */
    uint32_t start;               /* --start: PAM at the 5' end */
    int64_t  max_off_targets;     /* --max-off-targets, default -1 (unlimited) */
    const char* const* alt_pams;  /* -a */
    uint32_t n_alt_pams;
    uint32_t sam_scoring;         /* 0: specificity by the CSV rule (printer.hpp:244-300); 1: by the SAM rule (printer.hpp:115-170) */
    uint32_t iupac_pams;          /* --iupac-pam: read the pam column and alt_pams with IUPAC class letters (R, Y, S, W, K, M, B, D, H, V):
                                     a class matches its member bases, never a genome N.  0 (default): any letter but A, C, G, T, N never
                                     matches, as before.  (Appended field: callers built against the earlier, shorter struct must be rebuilt.) */
} gsx_params;

void gsx_params_default(gsx_params* p);

/* Per-guide and per-hit results, structure-of-arrays, valid until gsx_result_free().
 * Hits of guide g are hits [first_hit[g], first_hit[g] + n_hits[g]) in exactly the order of the reference's
 * off_targets vector (process.hpp:100-115): distance ascending, forward-index ("-" strand) hits before
 * reverse-index ("+") hits, std::set order of the match string, SA row ascending. */
typedef struct {
    size_t          n_guides;
    size_t          n_hits;
    uint32_t        n_dist;            /* mismatches + 1 */
    const uint8_t*  dropped;           /* [n_guides] 1 = removed by the threshold prefilter (prints nothing) */
    const uint64_t* first_hit;         /* [n_guides] */
    const uint32_t* n_hits_of;         /* [n_guides] */
    const float*    specificity;       /* [n_guides] float32, accumulated in reference order */
    const uint8_t*  perfect_match;     /* [n_guides] */
    const uint32_t* count_by_distance; /* [n_guides * n_dist] hits per distance before boundary filtering (SAM k<d>:i:) */
    /* per hit */
    const int64_t*  abs_pos;           /* sign/strand-encoded absolute coordinate (process.hpp:104,111) */
    const uint32_t* sa_row;            /* row of the suffix array (= the reference's bwt_position) */
    const int32_t*  chr;               /* chromosome index, -1 = boundary sentinel (structures.cxx:44-47): row is not printed */
    const uint32_t* pos1;              /* 1-based leftmost position on the + strand */
    const uint8_t*  strand;            /* '+' or '-' */
    const uint8_t*  distance;          /* mismatches */
    const uint8_t*  rna_bulges;
    const uint8_t*  dna_bulges;
    const uint8_t*  index_id;          /* 0 = forward index, 1 = reverse index */
    const float*    cfd;               /* calculate_cfd of the hit (printer.hpp:98-113) */
    const uint8_t*  counted;           /* 1 = inside the max_off_targets cut and resolved: contributes to specificity / is printed in CSV */
} gsx_result_view;

/* Work counters of one gsx_enumerate call (all devices summed). */
typedef struct {
    uint64_t nodes;            /* search-tree nodes expanded by the search kernel */
    uint64_t lookups;          /* occurrence-block lookups in the reference's unit (1 per jump-table line, 1-2 per node) */
    uint64_t matches;          /* SA intervals emitted (before de-duplication) */
    uint64_t hits;             /* located rows */
    uint64_t lf_steps;         /* LF steps of the locate kernel */
    uint64_t spills;           /* search-stack nodes spilled from shared memory to global memory */
    double   ms_search, ms_arrange, ms_locate, ms_score, ms_total_device;   /* CUDA-event times, max over devices */
    double   ms_h2d, ms_d2h;
    uint64_t launches;         /* kernels launched by this library for the call (all devices) */
    double   ms_sweep;         /* part of ms_search spent in the slice-major front end (0 if it did not run) */
    uint64_t seeds;            /* level-L nodes the front end handed to the tree search */
    double   ms_prepare;       /* host: guide validation / packing before the first device call */
    double   ms_wall;          /* host: wall time of the whole gsx_enumerate call */
    uint64_t sectors;          /* 32-byte index sectors the search kernels actually requested (= lookups when the front end is off) */
    uint64_t edited_guides;    /* bulge batches searched through edited guides (gsx_core.h variant_rewrite): how many of them; else 0 */
} gsx_counters;

/* ---- index ------------------------------------------------------------------------------------------- */
/* Opens <prefix>.forward / .reverse / .gs written by the reference's `guidescan index` (sdsl csa_wt<wt_huff<>,64,8192>;
 * layout: SURVEY.md App. B) or <prefix>.gsx / .gs written by gsx_index_build (both present: the more recently written), lays the
 * index out on the first of `devices`
 * (NULL / 0 => device 0; the derived arrays -- jump table, look-ahead lines, pattern summaries -- are computed there) and copies the
 * finished arrays to every further device, peer to peer.  A device named twice gives two job slots over one copy.
 * Replaces sdsl::load_from_file + genome_index construction, src/guidescan.cxx:186-211. */
int gsx_index_open(const char* prefix, const int* devices, int n_devices, gsx_index** out);
/* Builds the GPU index directly from a FASTA file on the device (suffix sorting on the GPU); replaces
 * do_index_cmd, src/guidescan.cxx:109-179.  If save_prefix != NULL also writes <save_prefix>.gsx + .gs. */
int gsx_index_build(const char* fasta_path, const char* save_prefix, const int* devices, int n_devices, gsx_index** out);
/* Same, from the raw upper-case concatenated genome already in host memory (what the reference keeps as
 * <fasta>.forward.dna, src/guidescan.cxx:127-141) and a chromosome table.  sa_shift: SA sample every 2^sa_shift rows
 * (6 = the reference's density 64). */
int gsx_index_build_text(const uint8_t* text, uint64_t length, const char* const* chr_names, const uint64_t* chr_lengths,
                         uint32_t n_chr, uint32_t sa_shift, const char* save_prefix, const int* devices, int n_devices,
                         gsx_index** out);
/* Writes the index in the reference's own format: <prefix>.forward / .reverse (sdsl csa_wt<wt_huff<>,64,8192>, byte for byte the
 * files the reference's `guidescan index` stores, src/guidescan.cxx:167-175, SURVEY.md App. B) and <prefix>.gs, so that an index
 * built here in seconds can be opened by the unmodified reference and by anything else that reads GuideScan2 indices.  Host work
 * only (all cores); needs SA samples at least every 64 rows (sa_shift <= 6). */
int gsx_index_save_reference_format(const gsx_index*, const char* prefix);
int gsx_index_close(gsx_index*);
uint64_t    gsx_index_genome_length(const gsx_index*);
uint32_t    gsx_index_n_chromosomes(const gsx_index*);
const char* gsx_index_chromosome_name(const gsx_index*, uint32_t i);
uint64_t    gsx_index_chromosome_length(const gsx_index*, uint32_t i);
uint64_t    gsx_index_device_bytes(const gsx_index*);
int         gsx_index_n_devices(const gsx_index*);
/* Seconds the open / build call spent: out[0] reading and converting the index files (or suffix sorting), out[1] upload and
 * derived arrays on the first device, out[2] replication to the other devices (peer copies over NVLink, all concurrently). */
/* 64-bit digest of everything the index holds on its slot-th device (computed there); replicas of one index give equal digests. */
int         gsx_index_device_checksum(const gsx_index*, int slot, uint64_t* out);
int         gsx_index_open_seconds(const gsx_index*, double out[3]);

/* Primitive queries (device-evaluated, for parity tests): occ of symbol c in BWT[0,i) = csa.rank_bwt(i,c)
 * (sdsl csa_wt.hpp:270-273) and SA[row] = csa[row] (csa_wt.hpp:333-346), batched. strand 0 = forward index. */
int gsx_index_rank(const gsx_index*, int strand, const uint64_t* rows, const char* syms, size_t n, uint64_t* out);
int gsx_index_locate(const gsx_index*, int strand, const uint64_t* rows, size_t n, uint64_t* out);
/* Host copies of what the index was built from, for cross-checking other implementations against the same index:
 * the BWT of text+'\0' as bytes (0 in the sentinel row; `out` holds genome_length + 1 bytes) and the SA samples
 * (SA[k << *sa_shift], ((n - 1) >> sa_shift) + 1 values). */
int gsx_index_export_bwt(const gsx_index*, int strand, uint8_t* out);
int gsx_index_export_sa_samples(const gsx_index*, int strand, uint32_t* out, uint64_t* n_samples, uint32_t* sa_shift);

/* ---- enumerate --------------------------------------------------------------------------------------- */
/* All guides, both strand indexes: search + locate + coordinates + CFD + specificity; results in host memory.
 * Guides are sharded over the index's devices (no collective; each device returns its own arena).
 * Inputs are borrowed for the duration of the call. */
int gsx_enumerate(const gsx_index*, const gsx_guide* guides, size_t n_guides, const gsx_params*, gsx_result** out);
/* The same call in two halves, for callers that pipeline batches: gsx_enumerate_start returns at once and the batch runs on a
 * library thread; gsx_enumerate_wait blocks until it is done, hands out the result (or the error) and releases the handle.
 * Calls in flight on the same device take turns from their first kernel to their last result copy, so what overlaps a running batch
 * is host work: packing the guides of the next one, formatting the result of the last one -- what the reference gets from N worker
 * threads behind one output mutex (src/guidescan.cxx:241-251, process.hpp:119-126).  `guides`, the strings they point to and `params` stay borrowed until
 * gsx_enumerate_wait returns. */
typedef struct gsx_pending gsx_pending;
int gsx_enumerate_start(const gsx_index*, const gsx_guide* guides, size_t n_guides, const gsx_params*, gsx_pending** out);
int gsx_enumerate_wait(gsx_pending*, gsx_result** out);
/* The arrays of the result.  With several devices every device returns its own part; the merged arrays of this view are built on the
 * first call (the library's own formatter, gsx_format_rows / gsx_enumerate_file, reads the parts in place and never needs them). */
int gsx_result_view_get(const gsx_result*, gsx_result_view* view);
int gsx_result_counters(const gsx_result*, gsx_counters* out);
/* The reference's match.sequence of hit `hit` complemented as it is printed (printer.hpp:232,264); buf >= 48 bytes. */
int gsx_result_match_sequence(const gsx_result*, size_t hit, char* buf, size_t buf_len);
void gsx_result_free(gsx_result*);

/* ---- text output (host C++; reproduces printer.hpp byte for byte) ------------------------------------ */
typedef struct {
    const char* id;
    const char* seq;
    const char* pam;
    int         sense_positive;      /* kmer.dir; only SAM uses it (FLAG 0/16, SEQ reverse-complemented) */
} gsx_guide_row;
/* format: 0 csv / 1 sam; complete: --mode complete.  Appends the rows of guides [g0, g1) to a malloc'ed buffer
 * (*buf, *len); the caller frees with gsx_free().  Headers: gsx_format_header(). */
int gsx_format_rows(const gsx_index*, const gsx_result*, const gsx_guide_row* rows, size_t g0, size_t g1,
                    const gsx_params*, int format_sam, int complete, char** buf, size_t* len);
int gsx_format_header(const gsx_index*, int format_sam, int complete, char** buf, size_t* len);
/* Whole-file convenience used by the CLI: guides CSV in -> CSV/SAM out (reference do_enumerate_cmd,
 * src/guidescan.cxx:181-258).  Returns the number of guides through *n_guides. */
int gsx_enumerate_file(const gsx_index*, const char* kmers_csv, const char* out_path, const gsx_params*,
                       int format_sam, int complete, size_t batch_guides, size_t* n_guides, gsx_counters* counters);
/* ---- guides CSV ingest (replaces genomics::kmer_producer, src/genomics/kmer.cxx:9-25 over include/csv.hpp) ----------------
 * The header must name the six columns id, sequence, pam, chromosome, position, sense (any order, nothing else); fields are
 * trimmed of spaces and tabs, there is no quoting; `position` is read and ignored, as downstream of the reference.  The file
 * is read whole and parsed by several host threads; rows keep file order.  Strings returned through gsx_guides_csv_row live
 * until gsx_guides_csv_close. */
typedef struct gsx_guide_table gsx_guide_table;
int  gsx_guides_csv_open(const char* path, gsx_guide_table** out, size_t* n_guides);
int  gsx_guides_csv_row(const gsx_guide_table*, size_t i, gsx_guide_row* row);
void gsx_guides_csv_close(gsx_guide_table*);
/* ---- genome-wide guide generation -------------------------------------------------------------------- */
/* What the reference's scripts/generate_kmers.py prints (reference scripts/generate_kmers.py:55-136): every k-mer next to an
 * occurrence of `pam` (N = any base) on either strand of every FASTA record of at least min_chr_length bases, as the guides
 * CSV that gsx_enumerate_file / `guidescan enumerate -f` reads.  `start` != 0: the PAM precedes the k-mer (--start).  The PAM
 * scan and the ordered compaction run on `device`; text identical to the script's.  *n_kmers (may be NULL) = rows written. */
int gsx_generate_kmers(const char* fasta_path, const char* out_csv_path, const char* pam, uint32_t kmer_length,
                       uint64_t min_chr_length, const char* prefix, int start, int device, uint64_t* n_kmers);
/* Generation and enumeration in one pass, without the guides CSV: writes byte for byte what gsx_generate_kmers(fasta_path, csv,
 * pam, kmer_length, min_chr_length, prefix, params->start) followed by gsx_enumerate_file(csv, out_path, ...) writes, for any
 * batch size and device list.  regions_bed != NULL keeps only the generated rows whose k bases lie inside one interval of the BED
 * file (0-based, half-open `chrom start end`; further columns, blank lines and `#` / `track` / `browser` lines are ignored); rows
 * keep the generator's order.  The index must be built from the same assembly: every FASTA record of at least min_chr_length
 * bases must be a chromosome of the index with the same length.  Options, FASTA and BED are checked before any device work
 * (GSX_ERR_ARG names the offending item).  The PAM scan runs on the index's first device, one chromosome at a time, taking that
 * device's turn like a call; host memory holds one chromosome, its sites and the batches in flight.  *n_guides = guides enumerated. */
int gsx_enumerate_genome(const gsx_index*, const char* fasta_path, const char* pam, uint32_t kmer_length, uint64_t min_chr_length,
                         const char* prefix, const char* regions_bed, const char* out_path, const gsx_params*, int format_sam,
                         int complete, size_t batch_guides, size_t* n_guides, gsx_counters* counters);

/* ---- SAM database decode ------------------------------------------------------------------------------ */
/* The off-targets of a database written by `enumerate --format sam --mode complete` (this library's or the original's), back as
 * rows: what scripts/decode_database.py of the original does, as the CSV that enumerate writes.  Per record: QNAME = guide id, SEQ
 * (reverse-complemented back when FLAG has 16) = protospacer + PAM column (its last pam_length characters), sp:f: = specificity
 * (copied as text); every position of the of:H: list becomes one row with its chromosome, position and strand (resolve_absolute),
 * the listed distance and the site's text from the genome, in record and list order.  Consecutive records of one QNAME are one guide:
 * the first is decoded, the others must carry the same list.  Each site is checked against its list: its mismatches to the guide
 * must be the listed distance, its PAM the guide's PAM column or one of alt_pams (of the column's length; N matches anything) --
 * a database written with bulges, with other PAMs or on another assembly fails with GSX_ERR_ARG naming the record and the site.
 * `fasta_path` is the assembly the database was computed on (its records must equal the SAM's @SQ lines); no index is needed.
 * complete: the columns of --mode complete (bulge columns 0), else succinct; with_cfd != 0 appends a `cfd` column (%.9g of the
 * float32 CFD the search computes).  regions_bed != NULL: only the records whose on-target site (RNAME:POS, len(SEQ) bases) lies
 * inside one BED interval.  Options, header, FASTA and BED are checked before any device work.  Runs on `device`; host memory holds
 * the genome and the batches in flight.  *n_guides = guides decoded, *n_rows = rows written (both may be NULL). */
int gsx_decode_database(const char* sam_path, const char* fasta_path, const char* out_path, uint32_t pam_length,
                        const char* const* alt_pams, uint32_t n_alt_pams, int complete, int with_cfd, const char* regions_bed,
                        int device, size_t* n_guides, size_t* n_rows);

void gsx_free(void*);

const char* gsx_last_error(void);
const char* gsx_version(void);     /* "2.0.0" -- reference include/version.hpp:2 */
int gsx_device_count(void);

#ifdef __cplusplus
}
#endif
#endif

"""ctypes binding of libgsx.so (include/gsx.h) -- the host-side mirror of the reference's per-guide pipeline
(`process_kmer_to_stream`, reference include/genomics/process.hpp:35-128) batched over guides.

There is no CPU path: if libgsx.so is missing this module raises at import, and every compute call fails with
GSX_ERR_NO_DEVICE when no CUDA device is present.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libgsx.so")
if not os.path.exists(LIB_PATH):
    raise ImportError("libgsx.so is not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
                      "(there is no fallback implementation)")
_L = C.CDLL(LIB_PATH)


class Guide(C.Structure):
    _fields_ = [("seq", C.c_char_p), ("pam", C.c_char_p)]


class Params(C.Structure):
    _fields_ = [("mismatches", C.c_uint32), ("rna_bulges", C.c_uint32), ("dna_bulges", C.c_uint32),
                ("max_bulge_size", C.c_uint32), ("threshold", C.c_int32), ("start", C.c_uint32),
                ("max_off_targets", C.c_int64), ("alt_pams", C.POINTER(C.c_char_p)), ("n_alt_pams", C.c_uint32),
                ("sam_scoring", C.c_uint32), ("iupac_pams", C.c_uint32)]


class ResultView(C.Structure):
    _fields_ = [("n_guides", C.c_size_t), ("n_hits", C.c_size_t), ("n_dist", C.c_uint32),
                ("dropped", C.POINTER(C.c_uint8)), ("first_hit", C.POINTER(C.c_uint64)), ("n_hits_of", C.POINTER(C.c_uint32)),
                ("specificity", C.POINTER(C.c_float)), ("perfect_match", C.POINTER(C.c_uint8)),
                ("count_by_distance", C.POINTER(C.c_uint32)),
                ("abs_pos", C.POINTER(C.c_int64)), ("sa_row", C.POINTER(C.c_uint32)), ("chr", C.POINTER(C.c_int32)),
                ("pos1", C.POINTER(C.c_uint32)), ("strand", C.POINTER(C.c_uint8)), ("distance", C.POINTER(C.c_uint8)),
                ("rna_bulges", C.POINTER(C.c_uint8)), ("dna_bulges", C.POINTER(C.c_uint8)), ("index_id", C.POINTER(C.c_uint8)),
                ("cfd", C.POINTER(C.c_float)), ("counted", C.POINTER(C.c_uint8))]


class Counters(C.Structure):
    _fields_ = [("nodes", C.c_uint64), ("lookups", C.c_uint64), ("matches", C.c_uint64), ("hits", C.c_uint64),
                ("lf_steps", C.c_uint64), ("spills", C.c_uint64), ("ms_search", C.c_double), ("ms_arrange", C.c_double),
                ("ms_locate", C.c_double), ("ms_score", C.c_double), ("ms_total_device", C.c_double),
                ("ms_h2d", C.c_double), ("ms_d2h", C.c_double), ("launches", C.c_uint64),
                ("ms_sweep", C.c_double), ("seeds", C.c_uint64), ("ms_prepare", C.c_double), ("ms_wall", C.c_double), ("sectors", C.c_uint64),
                ("edited_guides", C.c_uint64)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class GuideRow(C.Structure):
    _fields_ = [("id", C.c_char_p), ("seq", C.c_char_p), ("pam", C.c_char_p), ("sense_positive", C.c_int)]


EXPORTS = ["gsx_params_default", "gsx_index_open", "gsx_index_build", "gsx_index_build_text", "gsx_index_close",
           "gsx_index_genome_length",
           "gsx_index_n_chromosomes", "gsx_index_chromosome_name", "gsx_index_chromosome_length", "gsx_index_device_bytes",
           "gsx_index_n_devices", "gsx_index_save_reference_format", "gsx_index_open_seconds", "gsx_index_device_checksum", "gsx_enumerate_start", "gsx_enumerate_wait", "gsx_index_rank", "gsx_index_locate", "gsx_index_export_bwt", "gsx_index_export_sa_samples", "gsx_enumerate", "gsx_result_view_get",
           "gsx_result_counters", "gsx_result_match_sequence", "gsx_result_free", "gsx_format_rows", "gsx_format_header",
           "gsx_enumerate_file", "gsx_guides_csv_open", "gsx_guides_csv_row", "gsx_guides_csv_close", "gsx_generate_kmers", "gsx_enumerate_genome", "gsx_decode_database", "gsx_free", "gsx_last_error", "gsx_version", "gsx_device_count"]

_L.gsx_last_error.restype = C.c_char_p
_L.gsx_version.restype = C.c_char_p
_L.gsx_index_open.argtypes = [C.c_char_p, C.POINTER(C.c_int), C.c_int, C.POINTER(C.c_void_p)]
_L.gsx_index_save_reference_format.argtypes = [C.c_void_p, C.c_char_p]
_L.gsx_index_build.argtypes = [C.c_char_p, C.c_char_p, C.POINTER(C.c_int), C.c_int, C.POINTER(C.c_void_p)]
_L.gsx_index_build_text.argtypes = [C.c_void_p, C.c_uint64, C.POINTER(C.c_char_p), C.POINTER(C.c_uint64), C.c_uint32,
                                    C.c_uint32, C.c_char_p, C.POINTER(C.c_int), C.c_int, C.POINTER(C.c_void_p)]
_L.gsx_index_close.argtypes = [C.c_void_p]
_L.gsx_index_genome_length.restype = C.c_uint64
_L.gsx_index_genome_length.argtypes = [C.c_void_p]
_L.gsx_index_n_chromosomes.restype = C.c_uint32
_L.gsx_index_n_chromosomes.argtypes = [C.c_void_p]
_L.gsx_index_chromosome_name.restype = C.c_char_p
_L.gsx_index_chromosome_name.argtypes = [C.c_void_p, C.c_uint32]
_L.gsx_index_chromosome_length.restype = C.c_uint64
_L.gsx_index_chromosome_length.argtypes = [C.c_void_p, C.c_uint32]
_L.gsx_index_device_bytes.restype = C.c_uint64
_L.gsx_index_device_bytes.argtypes = [C.c_void_p]
_L.gsx_index_rank.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_char_p, C.c_size_t, C.c_void_p]
_L.gsx_index_locate.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]
_L.gsx_index_export_bwt.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
_L.gsx_index_export_sa_samples.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(C.c_uint32)]
_L.gsx_enumerate.argtypes = [C.c_void_p, C.POINTER(Guide), C.c_size_t, C.POINTER(Params), C.POINTER(C.c_void_p)]
_L.gsx_enumerate_start.argtypes = [C.c_void_p, C.POINTER(Guide), C.c_size_t, C.POINTER(Params), C.POINTER(C.c_void_p)]
_L.gsx_enumerate_wait.argtypes = [C.c_void_p, C.POINTER(C.c_void_p)]
_L.gsx_index_open_seconds.argtypes = [C.c_void_p, C.POINTER(C.c_double)]
_L.gsx_index_n_devices.argtypes = [C.c_void_p]
_L.gsx_index_device_checksum.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_uint64)]
_L.gsx_result_view_get.argtypes = [C.c_void_p, C.POINTER(ResultView)]
_L.gsx_result_counters.argtypes = [C.c_void_p, C.POINTER(Counters)]
_L.gsx_result_match_sequence.argtypes = [C.c_void_p, C.c_size_t, C.c_char_p, C.c_size_t]
_L.gsx_result_free.argtypes = [C.c_void_p]
_L.gsx_format_rows.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(GuideRow), C.c_size_t, C.c_size_t, C.POINTER(Params),
                               C.c_int, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]
_L.gsx_format_header.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]
_L.gsx_enumerate_file.argtypes = [C.c_void_p, C.c_char_p, C.c_char_p, C.POINTER(Params), C.c_int, C.c_int, C.c_size_t,
                                  C.POINTER(C.c_size_t), C.POINTER(Counters)]
_L.gsx_free.argtypes = [C.c_void_p]
_L.gsx_guides_csv_open.argtypes = [C.c_char_p, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]
_L.gsx_guides_csv_row.argtypes = [C.c_void_p, C.c_size_t, C.POINTER(GuideRow)]
_L.gsx_guides_csv_close.argtypes = [C.c_void_p]
_L.gsx_guides_csv_close.restype = None
_L.gsx_generate_kmers.argtypes = [C.c_char_p, C.c_char_p, C.c_char_p, C.c_uint32, C.c_uint64, C.c_char_p, C.c_int, C.c_int,
                                  C.POINTER(C.c_uint64)]
_L.gsx_enumerate_genome.argtypes = [C.c_void_p, C.c_char_p, C.c_char_p, C.c_uint32, C.c_uint64, C.c_char_p, C.c_char_p, C.c_char_p,
                                    C.POINTER(Params), C.c_int, C.c_int, C.c_size_t, C.POINTER(C.c_size_t), C.POINTER(Counters)]

_L.gsx_decode_database.argtypes = [C.c_char_p, C.c_char_p, C.c_char_p, C.c_uint32, C.POINTER(C.c_char_p), C.c_uint32, C.c_int, C.c_int,
                                   C.c_char_p, C.c_int, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]


class GsxError(RuntimeError):
    def __init__(self, code, where):
        self.code = code
        super().__init__("%s failed (status %d): %s" % (where, code, (_L.gsx_last_error() or b"").decode()))


def _ck(code, where):
    if code != 0:
        raise GsxError(code, where)


def device_count() -> int:
    return _L.gsx_device_count()


def generate_kmers(fasta: str, out_csv: str, pam="NGG", kmer_length=20, min_chr_length=0, prefix="", start=False, device=0) -> int:
    """scripts/generate_kmers.py of the reference (same options, same text), PAM scan on the GPU.  Returns the row count."""
    n = C.c_uint64()
    _ck(_L.gsx_generate_kmers(fasta.encode(), out_csv.encode(), pam.encode(), kmer_length, min_chr_length, prefix.encode(),
                              int(bool(start)), device, C.byref(n)), "gsx_generate_kmers")
    return n.value


def decode_database(sam: str, fasta: str, out: str, pam_length=3, alt_pams=(), mode="complete", cfd=False, regions=None, device=0):
    """The off-targets of a SAM complete database (`enumerate --format sam --mode complete`) back as enumerate's CSV rows, sites and
    CFD from `fasta` on the GPU (include/gsx.h gsx_decode_database).  Returns (guides decoded, rows written)."""
    arr = (C.c_char_p * max(1, len(alt_pams)))(*[a.encode() for a in alt_pams])
    ng, nr = C.c_size_t(), C.c_size_t()
    _ck(_L.gsx_decode_database(sam.encode(), fasta.encode(), out.encode(), pam_length, arr, len(alt_pams), int(mode == "complete"),
                               int(bool(cfd)), regions.encode() if regions else None, device, C.byref(ng), C.byref(nr)),
        "gsx_decode_database")
    return ng.value, nr.value


def make_params(mismatches=3, rna_bulges=0, dna_bulges=0, threshold=-1, start=False, max_off_targets=-1,
                alt_pams=(), sam_scoring=False, iupac_pams=False):
    """iupac_pams: read the guides' PAM column and alt_pams with IUPAC class letters (R, Y, S, W, K, M, B, D, H, V), each matching
    its member bases and never a genome N; off, any letter but A, C, G, T, N never matches."""
    p = Params()
    _L.gsx_params_default(C.byref(p))
    p.mismatches, p.rna_bulges, p.dna_bulges = mismatches, rna_bulges, dna_bulges
    p.threshold, p.start, p.max_off_targets = threshold, int(bool(start)), max_off_targets
    arr = (C.c_char_p * max(1, len(alt_pams)))(*[a.encode() for a in alt_pams])
    p.alt_pams = C.cast(arr, C.POINTER(C.c_char_p))
    p.n_alt_pams = len(alt_pams)
    p.sam_scoring = int(bool(sam_scoring))
    p.iupac_pams = int(bool(iupac_pams))
    p._keep = arr
    return p


class Result:
    def __init__(self, handle, index):
        self.h = handle
        self.index = index
        self.view = ResultView()
        _ck(_L.gsx_result_view_get(self.h, C.byref(self.view)), "gsx_result_view_get")

    def _arr(self, ptr, n, dtype):
        if n == 0:
            return np.zeros(0, dtype=dtype)
        return np.ctypeslib.as_array(ptr, shape=(n,)).view(dtype)

    @property
    def n_guides(self):
        return self.view.n_guides

    @property
    def n_hits(self):
        return self.view.n_hits

    def guide_arrays(self):
        v, n = self.view, self.view.n_guides
        return dict(dropped=self._arr(v.dropped, n, np.uint8), first_hit=self._arr(v.first_hit, n, np.uint64),
                    n_hits=self._arr(v.n_hits_of, n, np.uint32), specificity=self._arr(v.specificity, n, np.float32),
                    perfect_match=self._arr(v.perfect_match, n, np.uint8),
                    count_by_distance=self._arr(v.count_by_distance, n * v.n_dist, np.uint32).reshape(n, v.n_dist))

    def hit_arrays(self):
        v, n = self.view, self.view.n_hits
        return dict(abs_pos=self._arr(v.abs_pos, n, np.int64), sa_row=self._arr(v.sa_row, n, np.uint32),
                    chr=self._arr(v.chr, n, np.int32), pos1=self._arr(v.pos1, n, np.uint32), strand=self._arr(v.strand, n, np.uint8),
                    distance=self._arr(v.distance, n, np.uint8), rna=self._arr(v.rna_bulges, n, np.uint8),
                    dna=self._arr(v.dna_bulges, n, np.uint8), index_id=self._arr(v.index_id, n, np.uint8),
                    cfd=self._arr(v.cfd, n, np.float32), counted=self._arr(v.counted, n, np.uint8))

    def match_sequence(self, hit: int) -> str:
        buf = C.create_string_buffer(64)
        _ck(_L.gsx_result_match_sequence(self.h, hit, buf, 64), "gsx_result_match_sequence")
        return buf.value.decode()

    def counters(self) -> dict:
        c = Counters()
        _ck(_L.gsx_result_counters(self.h, C.byref(c)), "gsx_result_counters")
        return c.as_dict()

    def format(self, rows, params, fmt="csv", mode="complete") -> bytes:
        """rows: list of (id, seq, pam, sense_positive)"""
        arr = (GuideRow * max(1, len(rows)))()
        keep = []
        for i, (gid, seq, pam, pos) in enumerate(rows):
            b = (gid.encode(), seq.encode(), pam.encode())
            keep.append(b)
            arr[i] = GuideRow(b[0], b[1], b[2], int(pos))
        buf, ln = C.c_void_p(), C.c_size_t()
        _ck(_L.gsx_format_rows(self.index.h, self.h, arr, 0, len(rows), C.byref(params), int(fmt == "sam"),
                               int(mode == "complete"), C.byref(buf), C.byref(ln)), "gsx_format_rows")
        out = C.string_at(buf, ln.value)
        _L.gsx_free(buf)
        return out

    def close(self):
        if self.h:
            _L.gsx_result_free(self.h)
            self.h = None

    def __del__(self):
        self.close()


class Index:
    """Immutable GPU-resident genome index (both strands), replicated on `devices`."""

    def __init__(self, handle):
        self.h = handle

    @classmethod
    def open(cls, prefix: str, devices=None) -> "Index":
        h = C.c_void_p()
        dv = (C.c_int * len(devices))(*devices) if devices else None
        _ck(_L.gsx_index_open(prefix.encode(), dv, len(devices) if devices else 0, C.byref(h)), "gsx_index_open")
        return cls(h)

    @classmethod
    def build(cls, fasta: str, save_prefix: str | None = None, devices=None) -> "Index":
        h = C.c_void_p()
        dv = (C.c_int * len(devices))(*devices) if devices else None
        _ck(_L.gsx_index_build(fasta.encode(), save_prefix.encode() if save_prefix else None, dv,
                               len(devices) if devices else 0, C.byref(h)), "gsx_index_build")
        return cls(h)

    @classmethod
    def build_from_text(cls, text: np.ndarray, chroms, sa_shift: int = 6, save_prefix: str | None = None, devices=None) -> "Index":
        """text: uint8 upper-case concatenated genome (what the reference stores as <fasta>.forward.dna)"""
        text = np.ascontiguousarray(text, dtype=np.uint8)
        names = (C.c_char_p * len(chroms))(*[c[0].encode() for c in chroms])
        lens = (C.c_uint64 * len(chroms))(*[int(c[1]) for c in chroms])
        h = C.c_void_p()
        dv = (C.c_int * len(devices))(*devices) if devices else None
        _ck(_L.gsx_index_build_text(text.ctypes.data, text.size, names, lens, len(chroms), sa_shift,
                                    save_prefix.encode() if save_prefix else None, dv, len(devices) if devices else 0,
                                    C.byref(h)), "gsx_index_build_text")
        return cls(h)

    def close(self):
        if self.h:
            _L.gsx_index_close(self.h)
            self.h = None

    def __del__(self):
        self.close()

    @property
    def genome_length(self):
        return _L.gsx_index_genome_length(self.h)

    @property
    def device_bytes(self):
        return _L.gsx_index_device_bytes(self.h)

    @property
    def n_devices(self):
        return _L.gsx_index_n_devices(self.h)

    def device_checksum(self, slot: int) -> int:
        out = C.c_uint64()
        _ck(_L.gsx_index_device_checksum(self.h, slot, C.byref(out)), "gsx_index_device_checksum")
        return out.value

    def save_reference_format(self, prefix: str) -> None:
        """<prefix>.forward / .reverse / .gs as the reference's `guidescan index` writes them (src/guidescan.cxx:167-175)"""
        _ck(_L.gsx_index_save_reference_format(self.h, prefix.encode()), "gsx_index_save_reference_format")

    def open_seconds(self):
        """(files / suffix sorting, upload + derived arrays on the first device, replication to the other devices)"""
        out = (C.c_double * 3)()
        _ck(_L.gsx_index_open_seconds(self.h, out), "gsx_index_open_seconds")
        return tuple(out)

    def chromosomes(self):
        return [(_L.gsx_index_chromosome_name(self.h, i).decode(), _L.gsx_index_chromosome_length(self.h, i))
                for i in range(_L.gsx_index_n_chromosomes(self.h))]

    def rank(self, strand: int, rows, syms: str) -> np.ndarray:
        rows = np.ascontiguousarray(rows, dtype=np.uint64)
        out = np.zeros(len(rows), dtype=np.uint64)
        _ck(_L.gsx_index_rank(self.h, strand, rows.ctypes.data, syms.encode(), len(rows), out.ctypes.data), "gsx_index_rank")
        return out

    def locate(self, strand: int, rows) -> np.ndarray:
        rows = np.ascontiguousarray(rows, dtype=np.uint64)
        out = np.zeros(len(rows), dtype=np.uint64)
        _ck(_L.gsx_index_locate(self.h, strand, rows.ctypes.data, len(rows), out.ctypes.data), "gsx_index_locate")
        return out

    def export_bwt(self, strand: int) -> np.ndarray:
        out = np.empty(self.genome_length + 1, dtype=np.uint8)
        _ck(_L.gsx_index_export_bwt(self.h, strand, out.ctypes.data), "gsx_index_export_bwt")
        return out

    def export_sa_samples(self, strand: int):
        n, sh = C.c_uint64(), C.c_uint32()
        _ck(_L.gsx_index_export_sa_samples(self.h, strand, None, C.byref(n), C.byref(sh)), "gsx_index_export_sa_samples")
        out = np.empty(n.value, dtype=np.uint32)
        _ck(_L.gsx_index_export_sa_samples(self.h, strand, out.ctypes.data, C.byref(n), C.byref(sh)), "gsx_index_export_sa_samples")
        return out, sh.value

    def enumerate(self, guides, params) -> Result:
        """guides: sequence of (seq, pam) strings.  Mirrors genome_index::inexact_search + resolve + scoring for all guides."""
        n = len(guides)
        arr = (Guide * max(1, n))()
        keep = []
        for i, (seq, pam) in enumerate(guides):
            b = (seq.encode(), pam.encode())
            keep.append(b)
            arr[i] = Guide(b[0], b[1])
        h = C.c_void_p()
        _ck(_L.gsx_enumerate(self.h, arr, n, C.byref(params), C.byref(h)), "gsx_enumerate")
        return Result(h, self)

    def enumerate_raw(self, guide_array, n, params) -> Result:
        """pre-built ctypes Guide array (bench path: no per-call Python marshalling)"""
        h = C.c_void_p()
        _ck(_L.gsx_enumerate(self.h, guide_array, n, C.byref(params), C.byref(h)), "gsx_enumerate")
        return Result(h, self)

    def enumerate_start(self, guide_array, n, params):
        """first half of the two-slot form: returns a handle at once; the arguments must stay alive until enumerate_wait"""
        h = C.c_void_p()
        _ck(_L.gsx_enumerate_start(self.h, guide_array, n, C.byref(params), C.byref(h)), "gsx_enumerate_start")
        return h

    def enumerate_wait(self, pending) -> Result:
        h = C.c_void_p()
        _ck(_L.gsx_enumerate_wait(pending, C.byref(h)), "gsx_enumerate_wait")
        return Result(h, self)

    def header(self, fmt="csv", mode="complete") -> bytes:
        buf, ln = C.c_void_p(), C.c_size_t()
        _ck(_L.gsx_format_header(self.h, int(fmt == "sam"), int(mode == "complete"), C.byref(buf), C.byref(ln)), "gsx_format_header")
        out = C.string_at(buf, ln.value)
        _L.gsx_free(buf)
        return out

    def enumerate_file(self, kmers_csv: str, out_path: str, params, fmt="csv", mode="complete", batch_guides=0):
        n, c = C.c_size_t(), Counters()
        _ck(_L.gsx_enumerate_file(self.h, kmers_csv.encode(), out_path.encode(), C.byref(params), int(fmt == "sam"),
                                  int(mode == "complete"), batch_guides, C.byref(n), C.byref(c)), "gsx_enumerate_file")
        return n.value, c.as_dict()

    def enumerate_genome(self, fasta: str, out_path: str, params, pam="NGG", kmer_length=20, min_chr_length=0, prefix="",
                         regions=None, fmt="csv", mode="complete", batch_guides=0):
        """generate_kmers(fasta, ..., start=params.start) -> rows inside the BED file `regions` (None: all) -> enumerate_file, in
        one pass without the guides CSV.  Returns (guides, counters)."""
        n, c = C.c_size_t(), Counters()
        _ck(_L.gsx_enumerate_genome(self.h, fasta.encode(), pam.encode(), kmer_length, min_chr_length, prefix.encode(),
                                    regions.encode() if regions else None, out_path.encode(), C.byref(params), int(fmt == "sam"),
                                    int(mode == "complete"), batch_guides, C.byref(n), C.byref(c)), "gsx_enumerate_genome")
        return n.value, c.as_dict()


def read_guides_csv(path: str):
    """Rows of a guides CSV as (id, sequence, pam, sense_positive) through the library's own reader (host only, no GPU)."""
    h, n = C.c_void_p(), C.c_size_t()
    _ck(_L.gsx_guides_csv_open(path.encode(), C.byref(h), C.byref(n)), "gsx_guides_csv_open")
    try:
        out, row = [], GuideRow()
        for i in range(n.value):
            _ck(_L.gsx_guides_csv_row(h, i, C.byref(row)), "gsx_guides_csv_row")
            out.append((row.id.decode(), row.seq.decode(), row.pam.decode(), bool(row.sense_positive)))
        return out
    finally:
        _L.gsx_guides_csv_close(h)

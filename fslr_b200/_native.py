"""ctypes binding of include/fslr_b200.h (the C-ABI drop-in boundary).  No CPU fallback: importing works
without a GPU (so the symbols can be checked), but every compute entry point raises when the library or a
CUDA device is missing."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("FSLR_B200_LIB") or os.path.join(_HERE, "csrc", "libfslr_b200.so")   # (the variable: tuning builds)
MAX_FILLINGS = 64
N_STAGES = 14

SYMBOLS = ["fslrc_create", "fslrc_destroy", "fslrc_last_error", "fslrc_stage_name", "fslrc_version",
           "fslrc_cluster_device", "fslrc_cluster_host", "fslrc_filling_starts", "fslrc_mg_prepare", "fslrc_mg_pair", "fslrc_mg_partners", "fslrc_mg_replay",
           "fslrc_mg_finish", "fslrc_int_peak", "fslrc_launch_count", "fslrc_set_blocking_sync", "fslrc_choose_alignment_host",
           "fslrc_tsv_open", "fslrc_tsv_delete_false", "fslrc_tsv_chrom_name", "fslrc_tsv_read_names", "fslrc_tsv_write_cluster_bed", "fslrc_tsv_write_representative_bed",
           "fslrc_tsv_write_edges", "fslrc_tsv_close", "fslrc_set_edge_capture", "fslrc_edges",
           "fslrc_bam_open", "fslrc_bam_open_bgzf", "fslrc_bam_read_stream", "fslrc_bam_write_mappings_bed", "fslrc_bam_read_names", "fslrc_bam_close"]

ERRORS = {-1: "FSLRC_ERR_CUDA", -2: "FSLRC_ERR_ARG", -3: "FSLRC_ERR_ZERO_DIVISOR", -4: "FSLRC_ERR_TOO_MANY_FILLINGS",
          -5: "FSLRC_ERR_NALN_NOT_CONSTANT", -6: "FSLRC_ERR_OVERFLOW", -7: "FSLRC_ERR_RANGE", -8: "FSLRC_ERR_HASH_COLLISION"}
ERR_HASH_COLLISION = -8


class Table(C.Structure):
    _fields_ = [("n_rows", C.c_int64), ("n_reads", C.c_int64)] + \
               [(n, C.c_void_p) for n in ("read_id", "chrom", "rstart", "rend", "aln_size", "qstart", "qend", "n_alignments")] + \
               [("order", C.c_void_p), ("n_order", C.c_int64), ("chrom_u8", C.c_void_p), ("n_alignments_u16", C.c_void_p),
                ("rows_per_read_u8", C.c_void_p), ("aln_size_is_qspan", C.c_int64), ("rspan_i16", C.c_void_p),
                ("qstart_u16", C.c_void_p), ("qend_u16", C.c_void_p)]


class Params(C.Structure):
    _fields_ = [("overlap", C.c_double), ("qlen_c", C.c_double), ("naln_c", C.c_double),
                ("umax", C.c_int32 * (MAX_FILLINGS + 1)), ("edge_threshold", C.c_int64), ("n_chrom", C.c_int32),
                ("chrom_len", C.c_void_p), ("chrom_masked", C.c_void_p), ("mask_subtelomere", C.c_int32),
                ("subtel", C.c_int64)]


class Stats(C.Structure):
    _fields_ = [(n, C.c_int64) for n in ("n_fillings", "n_intervals", "n_query_reads", "band_pairs", "pair_tests",
                                          "relation_entries", "saturating_reads", "edges", "components", "clustered_reads",
                                          "partner_records")] + \
               [("no_clusters", C.c_int32), ("reserved", C.c_int32), ("stage_ms", C.c_float * N_STAGES)]

    def as_dict(self, lib=None):
        d = {n: int(getattr(self, n)) for n, _ in self._fields_[:11]}
        d["no_clusters"] = int(self.no_clusters)
        names = [lib.fslrc_stage_name(i).decode() for i in range(N_STAGES)] if lib is not None else list(range(N_STAGES))
        d["stage_ms"] = {names[i]: float(self.stage_ms[i]) for i in range(N_STAGES)}
        return d


class TsvInfo(C.Structure):
    _fields_ = [("n_rows", C.c_int64), ("n_reads", C.c_int64), ("n_chrom", C.c_int32), ("has_score", C.c_int32)] + \
               [(n, C.c_void_p) for n in ("read_id", "chrom", "rstart", "rend", "aln_size", "qstart", "qend", "n_alignments",
                                          "alignment_score")] + [("parse_ms", C.c_float), ("filter_ms", C.c_float)]


BAM_COLUMNS = ("read_id", "chrom", "rstart", "rend", "n_alignments", "aln_size", "qstart", "qend", "strand", "mapq", "qlen",
               "alignment_score", "short_anchor", "inferred_by_primer", "overlaps_region")


class BamInfo(C.Structure):
    _fields_ = [("n_records", C.c_int64), ("n_mapped", C.c_int64), ("n_reads", C.c_int64), ("n_rows", C.c_int64),
                ("n_chrom", C.c_int32), ("overlaps_as_float", C.c_int32)] + [(n, C.c_void_p) for n in BAM_COLUMNS] + \
               [("parse_ms", C.c_float), ("reserved", C.c_int32)]


class FslrError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("%s (%d): %s" % (ERRORS.get(code, "FSLRC_ERR"), code, msg))
        self.code = code


_lib = None


def load():
    """Load the shared library (raises if it has not been built: there is no fallback path)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError("fslr_b200: %s is missing — build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                           "or `make -C fslr_b200/csrc`; there is no CPU fallback" % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    vp, i64p = C.c_void_p, C.POINTER(C.c_int64)
    lib.fslrc_create.argtypes = [C.c_int, C.POINTER(vp)]
    lib.fslrc_destroy.argtypes = [vp]
    lib.fslrc_destroy.restype = None
    lib.fslrc_last_error.argtypes = [vp]
    lib.fslrc_last_error.restype = C.c_char_p
    lib.fslrc_stage_name.argtypes = [C.c_int]
    lib.fslrc_stage_name.restype = C.c_char_p
    lib.fslrc_version.restype = C.c_int
    for f in (lib.fslrc_cluster_device, lib.fslrc_cluster_host):
        f.argtypes = [vp, C.POINTER(Table), C.POINTER(Params), vp, vp, C.POINTER(Stats), vp]
    lib.fslrc_filling_starts.argtypes = [vp, C.POINTER(Table), vp, C.c_int64, i64p, vp]
    lib.fslrc_mg_prepare.argtypes = [vp, C.POINTER(Table), C.POINTER(Params), vp]
    lib.fslrc_mg_pair.argtypes = [vp, C.c_int, C.c_int, C.POINTER(vp), i64p]
    lib.fslrc_mg_partners.argtypes = [vp, C.c_int, C.c_int, C.POINTER(vp), i64p]
    lib.fslrc_mg_replay.argtypes = [vp, C.c_int, C.c_int, vp, C.c_int64, C.POINTER(vp), i64p]
    lib.fslrc_mg_finish.argtypes = [vp, vp, C.c_int64, vp, vp, C.POINTER(Stats)]
    lib.fslrc_int_peak.argtypes = [vp, C.POINTER(C.c_double)]
    lib.fslrc_choose_alignment_host.argtypes = [vp, C.c_int64, C.c_int64, C.c_int64, vp, vp, vp, vp, vp, vp]
    lib.fslrc_tsv_open.argtypes = [vp, vp, C.c_int64, C.c_uint64, C.POINTER(TsvInfo), vp]
    lib.fslrc_tsv_delete_false.argtypes = [vp, C.POINTER(TsvInfo), vp]
    lib.fslrc_tsv_chrom_name.argtypes = [vp, C.c_int32, C.c_char_p, C.c_int32]
    lib.fslrc_tsv_read_names.argtypes = [vp, vp, vp]
    lib.fslrc_tsv_write_cluster_bed.argtypes = [vp, vp, vp, vp, C.c_int64, i64p, vp]
    lib.fslrc_tsv_write_representative_bed.argtypes = [vp, vp, vp, vp, C.c_int64, i64p, vp]
    lib.fslrc_tsv_write_edges.argtypes = [vp, vp, C.c_int64, i64p, vp]
    lib.fslrc_set_edge_capture.argtypes = [vp, C.c_int]
    lib.fslrc_edges.argtypes = [vp, vp, vp, vp, C.c_int64, i64p, vp]
    lib.fslrc_tsv_close.argtypes = [vp]
    lib.fslrc_tsv_close.restype = None
    lib.fslrc_bam_open.argtypes = [vp, vp, C.c_int64, C.c_int64, C.c_int32, C.c_char_p, vp, C.c_int32, vp, vp, vp, C.c_int32, C.c_uint64,
                                   C.POINTER(BamInfo), vp]
    lib.fslrc_bam_open_bgzf.argtypes = lib.fslrc_bam_open.argtypes
    lib.fslrc_bam_read_stream.argtypes = [vp, vp, C.c_int64, i64p]
    lib.fslrc_bam_write_mappings_bed.argtypes = [vp, C.c_char_p, C.c_char_p, vp, C.c_int64, i64p, vp]
    lib.fslrc_bam_read_names.argtypes = [vp, vp, vp]
    lib.fslrc_bam_close.argtypes = [vp]
    lib.fslrc_bam_close.restype = None
    lib.fslrc_set_blocking_sync.argtypes = [vp, C.c_int]
    lib.fslrc_launch_count.argtypes = [vp]
    lib.fslrc_launch_count.restype = C.c_longlong
    _lib = lib
    return lib

"""ctypes binding of libmirfold.so (include/mirfold.h).  No fallback: import fails loudly if the
CUDA library has not been built (python __graft_entry__.py build, or make -C mir_prefer_b200/csrc)."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# MIRFOLD_LIB_PATH: load another build of the same library (kernel A/B experiments); never a fallback
LIB_PATH = os.environ.get("MIRFOLD_LIB_PATH") or os.path.join(_HERE, "libmirfold.so")


class MirfoldError(RuntimeError):
    def __init__(self, code, detail=""):
        self.code = code
        msg = "libmirfold error %d" % code
        if detail:
            msg += ": " + detail
        super().__init__(msg)


class Hit(C.Structure):
    _fields_ = [("start", C.c_int32), ("len", C.c_int32), ("mfe_dcal", C.c_int32), ("reserved", C.c_int32),
                ("ss_off", C.c_uint64)]


class Stats(C.Structure):
    _fields_ = [("ms_total", C.c_double), ("ms_h2d", C.c_double), ("ms_fill", C.c_double), ("ms_f3", C.c_double),
                ("ms_trace", C.c_double), ("ms_d2h", C.c_double), ("ms_device", C.c_double),
                ("nt", C.c_uint64), ("cells", C.c_uint64), ("tracebacks", C.c_uint64), ("kernel_launches", C.c_uint64),
                ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64), ("n_devices", C.c_int32), ("n_chunks", C.c_int32),
                ("fill_units", C.c_uint64)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class Result(C.Structure):
    _fields_ = [("nseq", C.c_uint32), ("reserved", C.c_uint32), ("nhits", C.c_uint64),
                ("hit_begin", C.POINTER(C.c_uint64)), ("hit_count", C.POINTER(C.c_uint32)), ("hits", C.POINTER(Hit)), ("ss_arena", C.c_void_p),
                ("ss_bytes", C.c_uint64), ("total_mfe_dcal", C.POINTER(C.c_int32)), ("stats", Stats)]


class Chunk(C.Structure):
    _fields_ = [("n_records", C.c_uint32), ("device", C.c_int32), ("record", C.POINTER(C.c_uint32)),
                ("hit_begin", C.POINTER(C.c_uint64)), ("hit_count", C.POINTER(C.c_uint32)),
                ("total_mfe_dcal", C.POINTER(C.c_int32)), ("nhits", C.c_uint64), ("hits", C.POINTER(Hit)),
                ("ss_arena", C.c_void_p), ("ss_bytes", C.c_uint64)]


CHUNK_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.POINTER(Chunk))


class Structure(C.Structure):
    _fields_ = [("rec", C.c_uint32), ("fold_start", C.c_int32), ("sstype", C.c_int32), ("len", C.c_int32),
                ("ss_off", C.c_uint64), ("norm_energy", C.c_double)]


class DuplexQuery(C.Structure):
    _fields_ = [("ss_off", C.c_uint64), ("ss_len", C.c_int32), ("fold_start", C.c_int32),
                ("mature_start", C.c_int32), ("mature_end", C.c_int32), ("region_start", C.c_int32),
                ("region_end", C.c_int32), ("strand", C.c_int32), ("reserved", C.c_int32)]


class DuplexVerdict(C.Structure):
    _fields_ = [("code", C.c_int32), ("star_start", C.c_int32), ("star_end", C.c_int32), ("fold_start", C.c_int32),
                ("fold_end", C.c_int32), ("star_ss_begin", C.c_int32), ("star_ss_end", C.c_int32),
                ("mature_ss_begin", C.c_int32), ("mature_ss_end", C.c_int32), ("prime5", C.c_int32),
                ("total_dots", C.c_int32), ("total_bps", C.c_int32)]


class Mature(C.Structure):
    _fields_ = [("start", C.c_int32), ("end", C.c_int32), ("strand", C.c_int32), ("depth", C.c_int32)]


class Region(C.Structure):
    _fields_ = [("start", C.c_int32), ("end", C.c_int32)]


class GenomeRegion(C.Structure):
    _fields_ = [("contig", C.c_int32), ("start", C.c_int32), ("end", C.c_int32), ("strand", C.c_int32)]


class Candidates(C.Structure):
    _fields_ = [("nseq", C.c_uint32), ("reserved", C.c_uint32), ("nstructs", C.c_uint64),
                ("struct_begin", C.POINTER(C.c_uint64)), ("struct_count", C.POINTER(C.c_uint32)),
                ("structs", C.POINTER(Structure)), ("ss_arena", C.c_void_p), ("ss_bytes", C.c_uint64),
                ("nverdicts", C.c_uint64), ("verdict_begin", C.POINTER(C.c_uint64)), ("verdict_count", C.POINTER(C.c_uint32)),
                ("verdicts", C.POINTER(DuplexVerdict)), ("verdict_mature", C.POINTER(C.c_uint32)), ("nhits", C.c_uint64),
                ("stats", Stats)]


class ShuffleStat(C.Structure):
    _fields_ = [("native_dcal", C.c_int32), ("n_le", C.c_uint32), ("sum_dcal", C.c_int64), ("sumsq_dcal", C.c_int64)]


class FillPlan(C.Structure):
    _fields_ = [("kernel", C.c_int32), ("stride", C.c_int32), ("tile_len", C.c_int32), ("tile_step", C.c_int32),
                ("n_units", C.c_int32), ("dmax", C.c_int32), ("band_cells", C.c_uint64)]


class Segment(C.Structure):
    _fields_ = [("tile_first", C.c_int32), ("tile_last", C.c_int32), ("halo_tiles", C.c_int32), ("row_first", C.c_int32),
                ("row_last", C.c_int32), ("reserved", C.c_int32), ("device_bytes", C.c_uint64)]


# every symbol include/mirfold.h declares
EXPORTS = ["mirfold_open", "mirfold_close", "mirfold_fold", "mirfold_fold_device", "mirfold_debug_matrices",
           "mirfold_free_result", "mirfold_strerror", "mirfold_last_error", "mirfold_version", "mirfold_duplex",
           "mirfold_duplex_fail_name", "mirfold_int_peak", "mirfold_format_records", "mirfold_free_text",
           "mirfold_classify", "mirfold_free_structures", "mirfold_fold_stream", "mirfold_batch_upload", "mirfold_batch_fold",
           "mirfold_batch_free", "mirfold_plan_shards", "mirfold_int_peak2", "mirfold_fold_candidates", "mirfold_free_candidates", "mirfold_fold_text", "mirfold_plan_fill_units",
           "mirfold_genome_upload", "mirfold_genome_free", "mirfold_fold_regions", "mirfold_fold_regions_stream",
           "mirfold_fold_candidates_regions", "mirfold_shuffle_test", "mirfold_shuffle_sequences", "mirfold_plan_segments"]

_lib = None


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError("libmirfold.so is not built (%s). Run `python __graft_entry__.py` or "
                          "`make -C mir_prefer_b200/csrc`. There is no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    vp = C.c_void_p
    lib.mirfold_open.argtypes = [C.POINTER(vp), C.POINTER(C.c_int), C.c_int, C.c_char_p]
    lib.mirfold_open.restype = C.c_int
    lib.mirfold_close.argtypes = [vp]
    lib.mirfold_close.restype = None
    lib.mirfold_fold.argtypes = [vp, C.c_void_p, C.POINTER(C.c_uint64), C.c_uint32, C.c_int, C.c_uint32,
                                 C.POINTER(C.POINTER(Result))]
    lib.mirfold_fold.restype = C.c_int
    lib.mirfold_fold_device.argtypes = [vp, C.c_void_p, C.c_void_p, C.POINTER(C.c_uint64), C.c_uint32, C.c_int,
                                        C.c_uint32, C.c_void_p, C.POINTER(C.POINTER(Result))]
    lib.mirfold_fold_device.restype = C.c_int
    lib.mirfold_debug_matrices.argtypes = [vp, C.c_char_p, C.c_uint32, C.c_int, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.mirfold_debug_matrices.restype = C.c_int
    lib.mirfold_format_records.argtypes = [C.POINTER(Result), C.c_void_p, C.POINTER(C.c_uint64), C.c_uint32,
                                           C.POINTER(C.c_void_p), C.POINTER(C.POINTER(C.c_uint64))]
    lib.mirfold_format_records.restype = C.c_int
    lib.mirfold_free_text.argtypes = [C.c_void_p, C.POINTER(C.c_uint64)]
    lib.mirfold_free_text.restype = None
    lib.mirfold_classify.argtypes = [C.POINTER(Result), C.c_int, C.c_int, C.POINTER(C.POINTER(Structure)),
                                     C.POINTER(C.c_uint64), C.POINTER(C.POINTER(C.c_uint64))]
    lib.mirfold_classify.restype = C.c_int
    lib.mirfold_free_structures.argtypes = [C.POINTER(Structure), C.POINTER(C.c_uint64)]
    lib.mirfold_free_structures.restype = None
    lib.mirfold_free_result.argtypes = [C.POINTER(Result)]
    lib.mirfold_free_result.restype = None
    lib.mirfold_strerror.argtypes = [C.c_int]
    lib.mirfold_strerror.restype = C.c_char_p
    lib.mirfold_last_error.argtypes = [vp]
    lib.mirfold_last_error.restype = C.c_char_p
    lib.mirfold_version.argtypes = []
    lib.mirfold_version.restype = C.c_char_p
    lib.mirfold_duplex.argtypes = [vp, C.c_void_p, C.c_uint64, C.POINTER(DuplexQuery), C.c_uint64,
                                   C.POINTER(DuplexVerdict)]
    lib.mirfold_duplex.restype = C.c_int
    lib.mirfold_duplex_fail_name.argtypes = [C.c_int]
    lib.mirfold_duplex_fail_name.restype = C.c_char_p
    lib.mirfold_int_peak.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    lib.mirfold_int_peak.restype = C.c_int
    lib.mirfold_int_peak2.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_double)]
    lib.mirfold_int_peak2.restype = C.c_int
    lib.mirfold_fold_stream.argtypes = [vp, C.c_void_p, C.POINTER(C.c_uint64), C.c_uint32, C.c_int, C.c_uint32, CHUNK_FN, C.c_void_p,
                                        C.POINTER(Stats)]
    lib.mirfold_fold_stream.restype = C.c_int
    lib.mirfold_batch_upload.argtypes = [vp, C.c_void_p, C.POINTER(C.c_uint64), C.c_uint32, C.c_int, C.POINTER(vp)]
    lib.mirfold_batch_upload.restype = C.c_int
    lib.mirfold_batch_fold.argtypes = [vp, vp, C.c_uint32, C.c_int, C.POINTER(C.POINTER(Result))]
    lib.mirfold_batch_fold.restype = C.c_int
    lib.mirfold_batch_free.argtypes = [vp]
    lib.mirfold_batch_free.restype = None
    lib.mirfold_plan_shards.argtypes = [C.POINTER(C.c_uint64), C.c_uint32, C.c_int, C.c_int, C.POINTER(C.c_uint32),
                                        C.POINTER(C.c_uint64)]
    lib.mirfold_plan_shards.restype = C.c_int
    if hasattr(lib, "mirfold_plan_fill_units"):
        lib.mirfold_plan_fill_units.argtypes = [C.c_uint32, C.c_int, C.POINTER(FillPlan)]
        lib.mirfold_plan_fill_units.restype = C.c_int
    if hasattr(lib, "mirfold_plan_segments"):
        lib.mirfold_plan_segments.argtypes = [C.c_uint32, C.c_int, C.c_uint64, C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32)]
        lib.mirfold_plan_segments.restype = C.c_int
    if os.environ.get("MIRFOLD_LIB_PATH") and not all(hasattr(lib, x) for x in ("mirfold_fold_candidates", "mirfold_fold_text")):
        _lib = lib      # an older A/B build of the library: the entry points below are not in it
        return lib
    lib.mirfold_fold_text.argtypes = [vp, C.c_char_p, C.c_uint64, C.c_int, C.c_uint32, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64)]
    lib.mirfold_fold_text.restype = C.c_int
    lib.mirfold_fold_candidates.argtypes = [vp, C.c_void_p, C.POINTER(C.c_uint64), C.c_uint32, C.c_int, C.c_uint32, C.c_void_p,
                                            C.c_void_p, C.POINTER(C.c_uint64), C.c_int, C.c_int, C.c_int, C.c_int,
                                            C.POINTER(C.POINTER(Candidates))]
    lib.mirfold_fold_candidates.restype = C.c_int
    lib.mirfold_free_candidates.argtypes = [C.POINTER(Candidates)]
    lib.mirfold_free_candidates.restype = None
    if hasattr(lib, "mirfold_genome_upload") or not os.environ.get("MIRFOLD_LIB_PATH"):   # an A/B build may predate genomes
        lib.mirfold_genome_upload.argtypes = [vp, C.c_void_p, C.POINTER(C.c_uint64), C.c_uint32, C.POINTER(vp)]
        lib.mirfold_genome_upload.restype = C.c_int
        lib.mirfold_genome_free.argtypes = [vp]
        lib.mirfold_genome_free.restype = None
        lib.mirfold_fold_regions.argtypes = [vp, vp, C.c_void_p, C.c_uint32, C.c_int, C.c_uint32, C.POINTER(C.POINTER(Result))]
        lib.mirfold_fold_regions.restype = C.c_int
        lib.mirfold_fold_regions_stream.argtypes = [vp, vp, C.c_void_p, C.c_uint32, C.c_int, C.c_uint32, CHUNK_FN, C.c_void_p,
                                                    C.POINTER(Stats)]
        lib.mirfold_fold_regions_stream.restype = C.c_int
        lib.mirfold_fold_candidates_regions.argtypes = [vp, vp, C.c_void_p, C.c_uint32, C.c_int, C.c_uint32, C.c_void_p,
                                                        C.POINTER(C.c_uint64), C.c_int, C.c_int, C.c_int, C.c_int,
                                                        C.POINTER(C.POINTER(Candidates))]
        lib.mirfold_fold_candidates_regions.restype = C.c_int
    if hasattr(lib, "mirfold_shuffle_test") or not os.environ.get("MIRFOLD_LIB_PATH"):   # an A/B build may predate the shuffle test
        lib.mirfold_shuffle_test.argtypes = [vp, C.c_void_p, C.POINTER(C.c_uint64), C.c_uint32, C.c_int, C.c_uint32, C.c_int,
                                             C.c_uint32, C.c_uint64, C.c_void_p, C.POINTER(Stats)]
        lib.mirfold_shuffle_test.restype = C.c_int
        lib.mirfold_shuffle_sequences.argtypes = [vp, C.c_void_p, C.POINTER(C.c_uint64), C.c_uint32, C.c_int, C.c_uint64, C.c_uint32,
                                                  C.c_void_p]
        lib.mirfold_shuffle_sequences.restype = C.c_int
    _lib = lib
    return lib

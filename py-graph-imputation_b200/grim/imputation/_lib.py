"""ctypes binding of libgrimb200.so / libgrimb200w.so (include/grimb200.h).

Two builds of the same ABI: libgrimb200.so packs a haplotype into a 64-bit key (GRIMB_KEY_WORDS
= 1; every table whose per-locus allele-id fields fit 63 bits), libgrimb200w.so into a 128-bit
key (GRIMB_KEY_WORDS = 2; wide 9-locus tables).  `load(kw)` picks one; Graph chooses kw from the
allele dictionary sizes.

There is no CPU path: if the CUDA library is missing or no device is present every entry point
raises.  The libraries are built in-tree by py-graph-imputation_b200/csrc/build.sh (or
__graft_entry__.build())."""
import ctypes as C
import os

MAX_LOCI = 9
MAX_ROWS = 16
MAX_BLOCKS = 9

ST_OK, ST_FAULT, ST_WORKSPACE, ST_SKIPPED, ST_NO_PHASES = 0, 2, 3, 4, 5
PLAN_NONE, PLAN_A, PLAN_B, PLAN_C = 0, 1, 2, 3
E_CAPACITY = -5
E_UNDEFINED = -6
ALL_POPS = 0xFFFF


class TableDesc(C.Structure):
    _fields_ = [
        ("n_loci", C.c_int32), ("n_pops", C.c_int32), ("n_full", C.c_int64),
        ("full_alleles", C.c_void_p), ("full_freqs", C.c_void_p),
        ("n_alleles", C.c_int32 * MAX_LOCI), ("key_bits", C.c_int32 * MAX_LOCI),
        ("last_parent_locus", C.c_int32), ("device", C.c_int32),
        ("label_masks", C.c_void_p), ("n_labels", C.c_int32), ("n_plan_a_labels", C.c_int32),
    ]


class TableInfo(C.Structure):
    _fields_ = [
        ("n_loci", C.c_int32), ("n_pops", C.c_int32), ("n_nodes", C.c_int64), ("n_full", C.c_int64),
        ("n_toplinks", C.c_int64), ("n_conn_edges", C.c_int64), ("n_slots", C.c_int64),
        ("device_bytes", C.c_int64),
    ]


class Config(C.Structure):
    _fields_ = [
        ("epsilon", C.c_double), ("factor_missing_pow", C.c_double * (MAX_LOCI + 1)),
        ("options_threshold", C.c_int64), ("max_haps_in_phase", C.c_int32), ("n_results", C.c_int32),
        ("n_pop_results", C.c_int32), ("planb", C.c_int32), ("output_umug", C.c_int32),
        ("output_pmug", C.c_int32), ("save_space", C.c_int32), ("compensated_sum", C.c_int32),
        ("n_rows", C.c_int32),
        ("row_blocks", C.c_int32 * MAX_ROWS), ("block_mask", (C.c_uint16 * MAX_BLOCKS) * MAX_ROWS),
        ("row_is_plan_a", C.c_uint8 * MAX_ROWS),
        ("hap_pop_pair", C.c_int32), ("em", C.c_int32), ("plan_a_only", C.c_int32),
        ("encounter_order", C.c_int32),
    ]


class Batch(C.Structure):
    _fields_ = [
        ("n_subjects", C.c_int64), ("typed_mask", C.c_void_p), ("counts", C.c_void_p),
        ("allele_off", C.c_void_p), ("alleles", C.c_void_p), ("n_alleles_total", C.c_int64),
        ("prior_index", C.c_void_p), ("priors", C.c_void_p), ("n_priors", C.c_int32),
        ("phase_mask", C.c_void_p), ("packed_keys", C.c_void_p), ("packed_flags", C.c_void_p),
    ]


SUBJECT_DTYPE = [
    ("status", "u1"), ("plan_umug", "u1"), ("plan_pmug", "u1"), ("reserved", "u1"),
    ("n_umug", "<u4"), ("n_pmug", "<u4"), ("n_umug_pops", "<u4"), ("n_pmug_pops", "<u4"),
    ("tot_umug", "<u4"), ("tot_pmug", "<u4"), ("pair_evals", "<u4"), ("hap_off", "<u8"), ("pop_off", "<u8"),
]  # GrimbSubjectResult, 48 bytes
HAP_ROW_DTYPE = [("a", "<u8"), ("b", "<u8"), ("prob", "<f8")]                    # GrimbHapRow, GRIMB_KEY_WORDS = 1
HAP_ROW_DTYPE_W = [("a", "<u8", (2,)), ("b", "<u8", (2,)), ("prob", "<f8")]      # GRIMB_KEY_WORDS = 2


def hap_row_dtype(kw=1):
    return HAP_ROW_DTYPE if kw == 1 else HAP_ROW_DTYPE_W
POP_ROW_DTYPE = [("pa", "<u2"), ("pb", "<u2"), ("pad", "<u4"), ("prob", "<f8")]


COMPACT_DTYPE = [("status", "u1"), ("kind_flags", "u1"), ("phases", "<u2"), ("off", "<u4"), ("total", "<f8")]  # GrimbCompact
KIND_GENERAL, KIND_SIMPLE, KIND_TYPED, KIND_WORDS, KIND_HAS_RESULTS = 0, 1, 2, 4, 8
NO_RECORD = 0xFFFFFFFF


class Results(C.Structure):
    _fields_ = [
        ("compact", C.c_void_p),
        ("words", C.c_void_p), ("word_capacity", C.c_int64),
        ("general", C.c_void_p), ("general_capacity", C.c_int64),
        ("hap_rows", C.c_void_p), ("hap_capacity", C.c_int64),
        ("pop_rows", C.c_void_p), ("pop_capacity", C.c_int64),
        ("totals", C.c_void_p),
    ]


class ResultArrays(object):
    """Host result buffers of one ABI call (numpy) + the GrimbResults struct pointing at them.
    totals: [words, general records, hap rows, pop rows, pair evaluations, handed to the general kernel,
    probes issued, probes answered, frequency vectors read]."""

    def __init__(self, n_subjects, kw=1, words=1024, general=1024, hap=1024, pop=1024):
        import numpy as np
        self.np = np
        self.kw = kw
        self.compact = np.zeros(max(1, n_subjects), dtype=COMPACT_DTYPE)
        self.totals = np.zeros(9, np.int64)
        self.caps = [max(16, int(words)), max(16, int(general)), max(16, int(hap)), max(16, int(pop))]
        self._alloc()

    def _alloc(self):
        np = self.np
        self.words = np.zeros(self.caps[0], np.uint64)
        self.general = np.zeros(self.caps[1], dtype=SUBJECT_DTYPE)
        self.hap_rows = np.zeros(self.caps[2], dtype=hap_row_dtype(self.kw))
        self.pop_rows = np.zeros(self.caps[3], dtype=POP_ROW_DTYPE)
        r = Results()
        r.compact = self.compact.ctypes.data
        r.words, r.word_capacity = self.words.ctypes.data, self.caps[0]
        r.general, r.general_capacity = self.general.ctypes.data, self.caps[1]
        r.hap_rows, r.hap_capacity = self.hap_rows.ctypes.data, self.caps[2]
        r.pop_rows, r.pop_capacity = self.pop_rows.ctypes.data, self.caps[3]
        r.totals = self.totals.ctypes.data
        self.struct = r

    def grow(self):
        """After GRIMB_E_CAPACITY: enlarge every array to what the call reported."""
        self.caps = [max(c, int(t)) for c, t in zip(self.caps, self.totals[:4])]
        self._alloc()


class TextDesc(C.Structure):
    _fields_ = [
        ("n_loci", C.c_int32), ("n_pops", C.c_int32),
        ("locus_names", C.POINTER(C.c_char_p)), ("allele_names", C.POINTER(C.c_char_p)),
        ("allele_counts", C.POINTER(C.c_int32)), ("pop_names", C.POINTER(C.c_char_p)),
        ("count_by_prob", C.POINTER(C.c_double)),
        ("alpha", C.c_double), ("eta", C.c_double), ("beta", C.c_double), ("gamma", C.c_double), ("delta", C.c_double),
        ("unk_priors_mr", C.c_int32), ("key_bits", C.c_int32 * MAX_LOCI), ("n_threads", C.c_int32),
        ("type_allowed", C.c_void_p),
    ]


class TextOut(C.Structure):
    _fields_ = [
        ("data", C.c_void_p * 6), ("size", C.c_int64 * 6),
        ("n_lines", C.c_int64), ("pair_evals", C.c_int64), ("workspace_retries", C.c_int64),
        ("plan_count", C.c_int64 * 4),
        ("seconds_tokenise", C.c_double), ("seconds_gpu", C.c_double), ("seconds_format", C.c_double),
    ]


class FileStats(C.Structure):
    _fields_ = [
        ("n_lines", C.c_int64), ("n_chunks", C.c_int64), ("in_bytes", C.c_int64), ("pair_evals", C.c_int64),
        ("workspace_retries", C.c_int64), ("plan_count", C.c_int64 * 4), ("out_bytes", C.c_int64 * 6),
        ("seconds_total", C.c_double), ("seconds_tokenise", C.c_double), ("seconds_gpu", C.c_double),
        ("seconds_format", C.c_double), ("seconds_write", C.c_double),
    ]


class Rows(C.Structure):
    """GrimbRows: ragged result rows decoded on the device (grimb_results_rows)."""
    _fields_ = [
        ("status", C.c_void_p), ("plan_umug", C.c_void_p), ("plan_pmug", C.c_void_p), ("flags", C.c_void_p),
        ("tot_umug", C.c_void_p), ("tot_pmug", C.c_void_p),
        ("off", C.c_void_p * 4), ("rows", C.c_void_p * 4), ("prob", C.c_void_p * 4), ("capacity", C.c_int64 * 4),
        ("totals", C.c_void_p), ("pmug_pairs", C.c_void_p),
    ]


ROW_KINDS = ("umug", "pmug", "umug_pops", "pmug_pops")   # GRIMB_ROWS_* order
ROWS_HAS_RESULTS, ROWS_MISS, ROWS_PROBLEM = 1, 2, 4

OUT_KEYS = ("umug", "umug_pops", "pmug", "pmug_pops", "miss", "problem")  # GRIMB_OUT_* order

_LIB = {}


def lib_path(kw=1):
    override = os.environ.get("GRIMB_LIB" if kw == 1 else "GRIMB_LIB_W")   # A/B runs of kernel variants
    if override:
        return override
    here = os.path.dirname(os.path.abspath(__file__))
    name = "libgrimb200.so" if kw == 1 else "libgrimb200w.so"
    return os.path.normpath(os.path.join(here, "..", "..", "csrc", name))


def load(kw=1):
    """Loads libgrimb200.so (kw = 1) or libgrimb200w.so (kw = 2), or raises: the product has no
    fallback."""
    if kw in _LIB:
        return _LIB[kw]
    path = lib_path(kw)
    if not os.path.exists(path):
        raise RuntimeError(
            "%s not built (%s): run py-graph-imputation_b200/csrc/build.sh; "
            "there is no CPU fallback" % (os.path.basename(path), path))
    lib = C.CDLL(path)
    lib.key_words = kw
    lib.grimb_abi_version.restype = C.c_int
    lib.grimb_last_error.restype = C.c_char_p
    lib.grimb_tables_build.argtypes = [C.POINTER(TableDesc), C.POINTER(C.c_void_p)]
    lib.grimb_tables_free.argtypes = [C.c_void_p]
    lib.grimb_tables_info.argtypes = [C.c_void_p, C.POINTER(TableInfo)]
    lib.grimb_tables_build_launches.argtypes = [C.c_void_p]
    lib.grimb_tables_build_launches.restype = C.c_int64
    lib.grimb_tables_export.argtypes = [C.c_void_p] + [C.c_void_p] * 10
    lib.grimb_tables_image_size.argtypes = [C.c_void_p, C.POINTER(C.c_int64)]
    lib.grimb_tables_image_ptr.argtypes = [C.c_void_p, C.POINTER(C.c_void_p)]
    lib.grimb_tables_image_copy.argtypes = [C.c_void_p, C.c_void_p]
    lib.grimb_tables_from_image.argtypes = [C.c_void_p, C.c_int64, C.c_int, C.POINTER(C.c_void_p)]
    lib.grimb_tables_build_ms.argtypes = [C.c_void_p]
    lib.grimb_tables_build_ms.restype = C.c_double
    lib.grimb_engine_create.argtypes = [C.c_void_p, C.c_int64, C.POINTER(C.c_void_p)]
    lib.grimb_engine_free.argtypes = [C.c_void_p]
    lib.grimb_engine_launches.argtypes = [C.c_void_p]
    lib.grimb_engine_launches.restype = C.c_int64
    lib.grimb_engine_kernel_ms.argtypes = [C.c_void_p, C.c_int]
    lib.grimb_engine_kernel_ms.restype = C.c_double
    lib.grimb_impute_device.argtypes = [C.c_void_p, C.POINTER(Config), C.POINTER(Batch), C.POINTER(Results), C.c_void_p]
    lib.grimb_impute_device_async.argtypes = [C.c_void_p, C.POINTER(Config), C.POINTER(Batch), C.POINTER(Results), C.c_void_p]
    lib.grimb_impute_finish.argtypes = [C.c_void_p, C.POINTER(Results)]
    lib.grimb_impute_host.argtypes = [C.c_void_p, C.POINTER(Config), C.POINTER(Batch), C.POINTER(Results)]
    lib.grimb_text_create.argtypes = [C.POINTER(TextDesc), C.POINTER(C.c_void_p)]
    lib.grimb_text_free.argtypes = [C.c_void_p]
    lib.grimb_text_tokenise.argtypes = [C.c_void_p, C.POINTER(Config), C.c_char_p, C.c_int64, C.c_int64, C.POINTER(Batch)]
    lib.grimb_text_format.argtypes = [C.c_void_p, C.POINTER(Config), C.POINTER(Results), C.POINTER(TextOut)]
    lib.grimb_impute_text.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.c_int32, C.POINTER(Config), C.c_char_p,
                                      C.c_int64, C.c_int64, C.POINTER(TextOut)]
    lib.grimb_impute_file.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.c_int32, C.POINTER(Config), C.c_char_p,
                                      C.c_int64, C.c_int64, C.c_int64, C.POINTER(C.c_char_p), C.c_int64,
                                      C.POINTER(TextOut), C.POINTER(FileStats)]
    lib.grimb_file_count_lines.argtypes = [C.c_char_p, C.c_int64, C.c_int64, C.c_int32, C.POINTER(C.c_int64),
                                           C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
    lib.grimb_file_write_at.argtypes = [C.c_char_p, C.c_int64, C.c_void_p, C.c_int64]
    lib.grimb_file_board_bytes.argtypes = [C.c_int64, C.c_int64]
    lib.grimb_file_board_bytes.restype = C.c_int64
    lib.grimb_impute_file_sharded.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.c_int32, C.POINTER(Config), C.c_char_p,
                                              C.POINTER(C.c_char_p), C.c_int64, C.c_int32, C.c_int32, C.c_char_p,
                                              C.POINTER(FileStats)]
    lib.grimb_batch_from_genotypes.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int32,
                                               C.c_void_p, C.POINTER(Batch), C.c_void_p]
    lib.grimb_batch_from_genotype_lists.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p,
                                                    C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.POINTER(Batch),
                                                    C.c_void_p]
    lib.grimb_results_rows.argtypes = [C.c_void_p, C.POINTER(Config), C.POINTER(Batch), C.POINTER(Results),
                                       C.POINTER(Rows), C.c_void_p]
    if lib.grimb_abi_version() != 5:
        raise RuntimeError("libgrimb200.so ABI mismatch")
    lib.grimb_struct_size.argtypes = [C.c_int32]
    lib.grimb_struct_size.restype = C.c_int64
    for which, ct in enumerate((Config, TableDesc, TextDesc, Batch, Results, TextOut, FileStats, TableInfo, Rows)):
        if lib.grimb_struct_size(which) != C.sizeof(ct):
            raise RuntimeError("libgrimb200.so: layout of %s differs from the binding (%d vs %d bytes)"
                               % (ct.__name__, lib.grimb_struct_size(which), C.sizeof(ct)))
    _LIB[kw] = lib
    return lib


def check(rc, what, lib=None):
    if rc != 0:
        msg = (lib or load()).grimb_last_error().decode("utf8", "replace")
        if rc == E_UNDEFINED:
            raise NotImplementedError("%s: %s" % (what, msg))
        raise RuntimeError("%s failed (%d): %s" % (what, rc, msg))


EXPORTED = [
    "grimb_abi_version", "grimb_last_error", "grimb_struct_size", "grimb_tables_build", "grimb_tables_free",
    "grimb_tables_info", "grimb_tables_build_launches", "grimb_tables_build_ms", "grimb_tables_export", "grimb_tables_image_size", "grimb_tables_image_ptr",
    "grimb_tables_image_copy", "grimb_tables_from_image", "grimb_engine_create", "grimb_engine_free", "grimb_engine_launches", "grimb_engine_kernel_ms",
    "grimb_impute_device", "grimb_impute_device_async", "grimb_impute_finish", "grimb_impute_host",
    "grimb_text_create", "grimb_text_free", "grimb_text_tokenise", "grimb_text_format", "grimb_impute_text",
    "grimb_impute_file", "grimb_file_count_lines", "grimb_file_write_at", "grimb_file_board_bytes",
    "grimb_impute_file_sharded", "grimb_batch_from_genotypes", "grimb_results_rows",
    "grimb_batch_from_genotype_lists",
]

"""ctypes binding of libkmerlr_b200.so (the C ABI declared in include/kmerlr_b200.h).

The shared library is built in-tree by ``__graft_entry__.build()`` / ``make -C kmerlr_b200/csrc``.
There is no CPU fallback: if the library is missing, or no sm_100 GPU is usable, calls raise.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "libkmerlr_b200.so")

OK, ERR_ARG, ERR_CUDA, ERR_INTERNAL, ERR_NOGPU = 0, 1, 2, 3, 4
TIE_GO118, TIE_INDEX = 0, 1
FLAG_SHARDED = 1
SUMMARY = {"": 0, "mean": 1, "product": 2, "min": 3, "max": 4}

# every symbol include/kmerlr_b200.h declares (tests check that the library exports all of them)
SYMBOLS = [
    "kmerlr_init", "kmerlr_shutdown", "kmerlr_last_error", "kmerlr_version", "kmerlr_last_device_ms",
    "kmerlr_launch_count", "kmerlr_option", "kmerlr_profile", "kmerlr_profile_read", "kmerlr_profile_dump", "kmerlr_comm_unique_id", "kmerlr_comm_init", "kmerlr_comm_destroy",
    "kmerlr_sequences_create", "kmerlr_sequences_from_fasta", "kmerlr_sequences_info", "kmerlr_sequences_names",
    "kmerlr_sequences_regions", "kmerlr_sequences_bases", "kmerlr_extract_resident", "kmerlr_extract", "kmerlr_matrix_info", "kmerlr_matrix_rows_global",
    "kmerlr_matrix_classes", "kmerlr_column_moments", "kmerlr_pair_moments", "kmerlr_matrix_transform", "kmerlr_matrix_rows", "kmerlr_matrix_set_labels", "kmerlr_matrix_from_csr",
    "kmerlr_matrix_subset",
    "kmerlr_free", "kmerlr_coeff_dim", "kmerlr_coeff_ind2sub", "kmerlr_coeff_sub2ind", "kmerlr_linear_pdf",
    "kmerlr_logpdf", "kmerlr_gradient", "kmerlr_loss", "kmerlr_class_weights", "kmerlr_select", "kmerlr_select_from_gradient", "kmerlr_reduce",
    "kmerlr_step_size", "kmerlr_proxgrad", "kmerlr_proxgrad_accel", "kmerlr_proxgrad_accel_full", "kmerlr_step_size_pairs", "kmerlr_proxgrad_pairs", "kmerlr_proxgrad_pairs_accel", "kmerlr_coordinate", "kmerlr_window_slots", "kmerlr_score_windows", "kmerlr_predict_windows",
    "kmerlr_score_windows_resident", "kmerlr_wiggle_records", "kmerlr_save_wiggle", "kmerlr_export_kmers", "kmerlr_class_name",
    "kmerlr_export_path", "kmerlr_export_trace",
]


class KmerLrError(RuntimeError):
    """Non-zero status from the C ABI (the Go shim turns these into log.Fatal / panic)."""

    def __init__(self, code, msg):
        super().__init__("kmerlr_b200 error %d: %s" % (code, msg))
        self.code = code


class Config(C.Structure):
    _fields_ = [(n, C.c_int32) for n in
                ("M", "N", "complement", "reverse", "revcomp", "binarize", "alphabet", "max_ambiguous")]


class Model(C.Structure):
    _fields_ = [("cfg", Config), ("n_classes", C.c_int64), ("class_k", C.POINTER(C.c_int32)),
                ("class_code", C.POINTER(C.c_uint64)), ("n_features", C.c_int64),
                ("features", C.POINTER(C.c_int32)), ("n_members", C.c_int64), ("theta", C.POINTER(C.c_double)),
                ("summary", C.c_int32)]


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise KmerLrError(ERR_NOGPU, "%s is missing: build it with __graft_entry__.build() "
                                     "(there is no CPU fallback)" % SO_PATH)
    L = C.CDLL(SO_PATH)
    vp, i64, i32, dbl, h = C.c_void_p, C.c_int64, C.c_int32, C.c_double, C.c_uint64
    ph, pi64, pdbl = C.POINTER(h), C.POINTER(i64), C.POINTER(dbl)
    L.kmerlr_init.argtypes = [C.c_int]
    L.kmerlr_last_error.restype = C.c_char_p
    L.kmerlr_last_device_ms.restype = dbl
    L.kmerlr_launch_count.restype = i64
    L.kmerlr_option.argtypes = [C.c_char_p, i64]
    L.kmerlr_profile.argtypes = [C.c_int]
    L.kmerlr_profile_read.argtypes = [C.c_char_p, pdbl, pi64]
    L.kmerlr_profile_dump.argtypes = [C.c_char_p, i64]
    L.kmerlr_comm_unique_id.argtypes = [vp]
    L.kmerlr_comm_init.argtypes = [C.c_int, C.c_int, vp]
    L.kmerlr_sequences_create.argtypes = [vp, vp, i64, ph]
    L.kmerlr_sequences_from_fasta.argtypes = [vp, vp, i64, vp, ph]
    L.kmerlr_sequences_info.argtypes = [h, pi64, pi64, vp]
    L.kmerlr_sequences_names.argtypes = [h, vp, i64, vp]
    L.kmerlr_sequences_regions.argtypes = [h, vp, vp, vp, i64, ph]
    L.kmerlr_sequences_bases.argtypes = [h, vp]
    L.kmerlr_extract_resident.argtypes = [C.POINTER(Config), h, vp, vp, i64, vp, i64, C.c_int, ph]
    L.kmerlr_extract.argtypes = [C.POINTER(Config), vp, vp, i64, vp, vp, i64, vp, i64, C.c_int, ph]
    L.kmerlr_matrix_info.argtypes = [h, pi64, pi64, pi64, pi64]
    L.kmerlr_matrix_rows_global.argtypes = [h, pi64]
    L.kmerlr_matrix_classes.argtypes = [h, vp, vp]
    L.kmerlr_matrix_rows.argtypes = [h, vp, vp, vp]
    L.kmerlr_column_moments.argtypes = [h, vp, vp, vp, vp]
    L.kmerlr_pair_moments.argtypes = [h, vp, vp, vp, vp]
    L.kmerlr_matrix_transform.argtypes = [h, vp, vp, i64, ph]
    L.kmerlr_matrix_set_labels.argtypes = [h, vp, i64]
    L.kmerlr_matrix_from_csr.argtypes = [i64, i64, vp, vp, vp, C.c_int, ph]
    L.kmerlr_matrix_subset.argtypes = [h, vp, i64, ph]
    L.kmerlr_free.argtypes = [h]
    L.kmerlr_coeff_dim.restype = i64
    L.kmerlr_coeff_dim.argtypes = [i64]
    L.kmerlr_coeff_ind2sub.restype = i64
    L.kmerlr_coeff_ind2sub.argtypes = [i64, i64, i64]
    L.kmerlr_coeff_sub2ind.restype = None
    L.kmerlr_coeff_sub2ind.argtypes = [i64, i64, pi64, pi64]
    L.kmerlr_linear_pdf.argtypes = [h, vp, i64, C.c_int, vp]
    L.kmerlr_logpdf.argtypes = [h, vp, i64, C.c_int, vp]
    L.kmerlr_gradient.argtypes = [h, vp, i64, vp, dbl, C.c_int, vp]
    L.kmerlr_loss.argtypes = [h, vp, i64, vp, dbl, C.c_int, pdbl]
    L.kmerlr_class_weights.argtypes = [h, vp]
    L.kmerlr_select.argtypes = [h, vp, C.c_int, i64, dbl, vp, vp, i64, C.c_int, dbl, dbl, vp, i64, pdbl, pi64,
                                C.POINTER(C.c_int), vp]
    L.kmerlr_select_from_gradient.argtypes = [vp, i64, i64, vp, vp, i64, C.c_int, dbl, dbl, vp, pdbl, pi64, C.POINTER(C.c_int)]
    L.kmerlr_reduce.argtypes = [h, vp, i64, ph]
    L.kmerlr_step_size.argtypes = [h, dbl, dbl, pdbl]
    L.kmerlr_proxgrad.argtypes = [h, vp, i64, vp, dbl, dbl, dbl, dbl, dbl, i64, vp, pi64, pdbl]
    L.kmerlr_proxgrad_accel.argtypes = [h, vp, vp, pdbl, i64, vp, dbl, dbl, dbl, dbl, dbl, i64, vp, pi64, pdbl, pi64]
    L.kmerlr_proxgrad_accel_full.argtypes = [h, vp, vp, pdbl, i64, vp, dbl, dbl, dbl, dbl, dbl, i64, vp, pi64, pdbl, pi64]
    L.kmerlr_step_size_pairs.argtypes = [h, dbl, dbl, pdbl]
    L.kmerlr_proxgrad_pairs.argtypes = [h, vp, i64, vp, dbl, dbl, dbl, dbl, dbl, i64, vp, pi64, pdbl]
    L.kmerlr_proxgrad_pairs_accel.argtypes = [h, vp, vp, pdbl, i64, vp, dbl, dbl, dbl, dbl, dbl, i64, vp, pi64, pdbl, pi64]
    L.kmerlr_coordinate.argtypes = [h, vp, i64, vp, dbl, dbl, dbl, dbl, i64, vp, pi64, pdbl]
    L.kmerlr_window_slots.restype = i64
    L.kmerlr_window_slots.argtypes = [i64, i64, i64]
    L.kmerlr_score_windows.argtypes = [C.POINTER(Model), C.c_int, vp, vp, i64, i64, i64, vp]
    L.kmerlr_predict_windows.argtypes = [C.POINTER(Model), vp, vp, i64, i64, i64, vp]
    L.kmerlr_score_windows_resident.argtypes = [C.POINTER(Model), C.c_int, h, i64, i64, vp, ph]
    ppc = C.POINTER(C.c_char_p)
    L.kmerlr_wiggle_records.argtypes = [vp, i64, vp, pi64]
    L.kmerlr_save_wiggle.argtypes = [C.c_char_p, C.c_char_p, i64, ppc, vp, vp, vp, h, i64, i64]
    L.kmerlr_export_kmers.argtypes = [h, C.POINTER(Config), C.c_char_p, C.c_int]
    L.kmerlr_class_name.argtypes = [C.POINTER(Config), i32, C.c_uint64, C.c_char_p, i64]
    L.kmerlr_export_path.argtypes = [C.c_char_p, i64, vp, vp, vp, vp, vp]
    L.kmerlr_export_trace.argtypes = [C.c_char_p, i64, vp, vp, vp, vp, vp, vp]
    _lib = L
    return L


def check(rc):
    if rc != OK:
        raise KmerLrError(rc, lib().kmerlr_last_error().decode(errors="replace"))

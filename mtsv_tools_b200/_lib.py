"""ctypes loader of libmtsv_b200.so (the C ABI declared in include/mtsv_b200.h)."""
import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
# (MTSV_B200_LIB: an alternative build of the same library, for A/B measurements of compile-time knobs)
LIB_PATH = os.environ.get("MTSV_B200_LIB") or os.path.join(_HERE, "libmtsv_b200.so")
_LIB = None

E_NAMES = {0: "OK", -1: "EINVAL", -2: "EIO", -3: "EFORMAT", -4: "ENODEVICE", -5: "ECUDA", -6: "ENOMEM",
           -7: "ELIMIT"}
N_STAGES = 12
STAGE_NAMES = ["prep", "seed_search", "seed_select", "locate", "sort", "coalesce", "rank", "verify",
               "emit", "copy"]


class LibraryError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("mtsv_b200 error %s (%d): %s" % (E_NAMES.get(code, "?"), code, msg))
        self.code = code


class HitStruct(C.Structure):
    _fields_ = [("tax_id", C.c_uint32), ("gi", C.c_uint32), ("offset", C.c_uint64),
                ("edit", C.c_uint32), ("reserved", C.c_uint32)]


class TaxHitStruct(C.Structure):
    _fields_ = [("tax_id", C.c_uint32), ("edit", C.c_uint32)]


class BinStruct(C.Structure):
    _fields_ = [("gi", C.c_uint32), ("tax_id", C.c_uint32), ("start", C.c_uint64), ("end", C.c_uint64)]


class ParamsStruct(C.Structure):
    _fields_ = [("edit_rate", C.c_double), ("seed_size", C.c_uint32), ("seed_gap", C.c_uint32),
                ("min_seed", C.c_double), ("max_hits", C.c_uint64), ("tune_max_hits", C.c_uint64),
                ("max_candidates", C.c_int64), ("max_assignments", C.c_int64),
                ("strands", C.c_uint32), ("reserved", C.c_uint32)]


class OptsStruct(C.Structure):
    _fields_ = [("sa_rate", C.c_uint32), ("ktab_k", C.c_uint32), ("max_batch_hits", C.c_uint64),
                ("batch_reads", C.c_uint32), ("reserved", C.c_uint32)]


class InfoStruct(C.Structure):
    _fields_ = [("text_len", C.c_uint64), ("n_bins", C.c_uint64), ("file_sa_rate", C.c_uint64),
                ("device_sa_rate", C.c_uint32), ("ktab_k", C.c_uint32), ("device_bytes", C.c_uint64),
                ("dollar_row", C.c_uint64), ("load_seconds", C.c_double),
                ("relayout_seconds", C.c_double), ("build_seconds", C.c_double)]


class StatsStruct(C.Structure):
    _fields_ = [("ms", C.c_float * N_STAGES), ("launches", C.c_uint64 * N_STAGES),
                ("n_queries", C.c_uint64), ("n_seed_slots", C.c_uint64), ("n_seed_hits", C.c_uint64),
                ("n_candidates", C.c_uint64), ("n_hits", C.c_uint64), ("window_bytes", C.c_uint64),
                ("rank_queries", C.c_uint64), ("n_sub_batches", C.c_uint64), ("h2d_bytes", C.c_uint64),
                ("n_reads_over_limit", C.c_uint64), ("n_strands_over_hits", C.c_uint64)]


# every symbol include/mtsv_b200.h declares
EXPORTS = [
    "mtsvgpu_index_open", "mtsvgpu_index_from_parts", "mtsvgpu_index_build", "mtsvgpu_index_write", "mtsvgpu_index_export", "mtsvgpu_suffix_array", "mtsvgpu_index_close", "mtsvgpu_index_get_info",
    "mtsvgpu_bin_batch", "mtsvgpu_bin_batch_pinned", "mtsvgpu_bin_batch_device", "mtsvgpu_bin_batch_packed", "mtsvgpu_assign_batch_device", "mtsvgpu_assign_batch_pinned", "mtsvgpu_assign_batch_packed", "mtsvgpu_packed_size", "mtsvgpu_pack_reads", "mtsvgpu_pack_read", "mtsvgpu_host_alloc", "mtsvgpu_host_free", "mtsvgpu_last_batch_stats", "mtsvgpu_set_stream",
    "mtsvgpu_set_profiling", "mtsvgpu_backward_search", "mtsvgpu_locate", "mtsvgpu_edit_distance",
    "mtsvgpu_collapse_device", "mtsvgpu_collapse_device_taxid_gi", "mtsvgpu_device_free", "mtsvgpu_comm_create", "mtsvgpu_comm_connect", "mtsvgpu_comm_destroy", "mtsvgpu_bin_batch_chunked", "mtsvgpu_free", "mtsvgpu_last_error", "mtsvgpu_launch_count", "mtsvgpu_version",
]


def build_library(force=False):
    """Compile csrc/*.cu for sm_100a into libmtsv_b200.so (nvcc cross-compiles without a GPU)."""
    csrc = os.path.join(_HERE, "csrc")
    args = ["make", "-s", "-C", csrc]
    if force:
        args.append("-B")
    subprocess.check_call(args)
    return LIB_PATH


def load_library():
    """Load the CUDA library or fail loudly — there is no other implementation behind this package."""
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(LIB_PATH):
        raise LibraryError(-4, "%s is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                               "(needs nvcc); there is no CPU fallback" % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    vp, u64p = C.c_void_p, C.POINTER(C.c_uint64)
    L.mtsvgpu_version.restype = C.c_char_p
    L.mtsvgpu_last_error.restype = C.c_char_p
    L.mtsvgpu_launch_count.restype = C.c_uint64
    L.mtsvgpu_free.argtypes = [vp]
    L.mtsvgpu_index_open.argtypes = [C.c_char_p, C.c_int, C.POINTER(OptsStruct), C.POINTER(vp)]
    L.mtsvgpu_index_from_parts.argtypes = [vp, C.c_uint64, vp, C.c_uint64, vp, vp, C.c_uint64,
                                           C.c_uint64, C.c_int, C.POINTER(OptsStruct), C.POINTER(vp)]
    L.mtsvgpu_index_build.argtypes = [vp, vp, vp, vp, C.c_uint64, C.c_int, C.POINTER(OptsStruct), C.POINTER(vp)]
    L.mtsvgpu_index_write.argtypes = [vp, C.c_char_p, C.c_uint32, C.c_uint32]
    L.mtsvgpu_index_export.argtypes = [vp, vp, vp, vp, C.c_uint32]
    L.mtsvgpu_suffix_array.argtypes = [C.c_int, vp, C.c_uint64, vp, vp]
    L.mtsvgpu_index_close.argtypes = [vp]
    L.mtsvgpu_index_get_info.argtypes = [vp, C.POINTER(InfoStruct)]
    L.mtsvgpu_bin_batch.argtypes = [vp, vp, vp, C.c_uint64, C.POINTER(ParamsStruct),
                                    C.POINTER(C.POINTER(HitStruct)), C.POINTER(u64p)]
    L.mtsvgpu_bin_batch_pinned.argtypes = [vp, vp, vp, C.c_uint64, C.POINTER(ParamsStruct),
                                           C.POINTER(vp), C.POINTER(vp), u64p]
    L.mtsvgpu_bin_batch_device.argtypes = [vp, vp, vp, C.c_uint64, C.POINTER(ParamsStruct),
                                           C.POINTER(vp), C.POINTER(vp), u64p]
    L.mtsvgpu_bin_batch_packed.argtypes = [vp, vp, C.c_uint64, vp, C.c_uint64, C.POINTER(ParamsStruct),
                                           C.POINTER(vp), C.POINTER(vp), u64p]
    L.mtsvgpu_assign_batch_device.argtypes = L.mtsvgpu_bin_batch_device.argtypes
    L.mtsvgpu_assign_batch_pinned.argtypes = L.mtsvgpu_bin_batch_pinned.argtypes
    L.mtsvgpu_assign_batch_packed.argtypes = L.mtsvgpu_bin_batch_packed.argtypes
    L.mtsvgpu_packed_size.restype = C.c_uint64
    L.mtsvgpu_packed_size.argtypes = [vp, C.c_uint64]
    L.mtsvgpu_pack_reads.argtypes = [vp, vp, C.c_uint64, vp, C.c_uint64, u64p, C.c_int]
    L.mtsvgpu_pack_read.argtypes = [vp, C.c_uint32, vp]
    L.mtsvgpu_host_alloc.restype = vp
    L.mtsvgpu_host_alloc.argtypes = [C.c_uint64]
    L.mtsvgpu_host_free.argtypes = [vp]
    L.mtsvgpu_last_batch_stats.argtypes = [vp, C.POINTER(StatsStruct)]
    L.mtsvgpu_set_stream.argtypes = [vp, vp]
    L.mtsvgpu_set_profiling.argtypes = [vp, C.c_int]
    L.mtsvgpu_backward_search.argtypes = [vp, vp, C.c_uint32, C.c_uint64, vp, vp]
    L.mtsvgpu_locate.argtypes = [vp, vp, C.c_uint64, vp]
    L.mtsvgpu_collapse_device.argtypes = [C.c_int, vp, C.c_uint32, C.POINTER(vp), C.POINTER(vp), C.c_uint64,
                                          C.POINTER(vp), C.POINTER(vp), u64p]
    L.mtsvgpu_collapse_device_taxid_gi.argtypes = L.mtsvgpu_collapse_device.argtypes
    L.mtsvgpu_device_free.argtypes = [vp]
    L.mtsvgpu_comm_create.argtypes = [C.c_int, C.c_uint32, C.c_uint32, C.c_uint64, C.c_uint64, C.POINTER(vp), vp]
    L.mtsvgpu_comm_connect.argtypes = [vp, vp]
    L.mtsvgpu_comm_destroy.argtypes = [vp]
    L.mtsvgpu_bin_batch_chunked.argtypes = [vp, vp, vp, vp, C.c_uint64, C.POINTER(ParamsStruct), u64p, u64p,
                                            C.POINTER(vp), C.POINTER(vp), u64p]
    L.mtsvgpu_edit_distance.argtypes = [C.c_int, vp, vp, vp, vp, C.c_uint64, vp]
    _LIB = L
    return L


def check(rc):
    if rc != 0:
        raise LibraryError(rc, load_library().mtsvgpu_last_error().decode(errors="replace"))

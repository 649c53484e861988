"""ctypes loader for libtblup_b200.so (the C-ABI declared in include/tblup_b200.h).

The library is built in-tree by ``__graft_entry__.build()`` / ``make -C tblup_b200/csrc``.  There is no
CPU fallback: if the shared object is missing or a CUDA device is absent, calls fail loudly.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("TBLUP_B200_LIB") or os.path.join(_HERE, "libtblup_b200.so")   # (override: A/B of library builds)

# every symbol include/tblup_b200.h declares: name -> (restype, argtypes)
_i32p = C.POINTER(C.c_int32)
_i64p = C.POINTER(C.c_int64)
_f64p = C.POINTER(C.c_double)
SYMBOLS = {
    "tb_abi_version": (C.c_int, []),
    "tb_last_error": (C.c_char_p, [C.c_void_p]),
    "tb_create": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_void_p)]),
    "tb_create_ex": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int,
                               C.POINTER(C.c_void_p)]),
    "tb_storage_info": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "tb_destroy": (C.c_int, [C.c_void_p]),
    "tb_clone": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p)]),
    "tb_set_rowset": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int]),
    "tb_pack_index_lists": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_void_p, C.c_void_p,
                                      C.POINTER(C.c_int64)]),
    "tb_stage_genomes": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    "tb_eval_staged": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_double, C.c_int, C.c_void_p, C.c_int]),
    "tb_eval": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_double, C.c_int,
                          C.c_void_p]),
    "tb_gram_debug": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "tb_debug_fetch": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_size_t]),
    "tb_set_option": (C.c_int, [C.c_void_p, C.c_char_p, C.c_longlong]),
    "tb_get_info": (C.c_int, [C.c_void_p, C.c_char_p, C.POINTER(C.c_longlong)]),
    "tb_staged_offsets": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int]),
    "tb_stage_times": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "tb_launch_count": (C.c_uint64, [C.c_void_p]),
    "tb_reset_counters": (C.c_int, [C.c_void_p]),
    "tb_last_wave": (C.c_int, [C.c_void_p]),
    "tb_last_precision": (C.c_int, [C.c_void_p]),
    "tb_de_init": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_uint64]),
    "tb_de_evaluate": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_double, C.c_int]),
    "tb_de_step": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_double, C.c_int, C.c_double, C.c_double, C.c_int,
                             C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    "tb_de_step_begin": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_double, C.c_int, C.c_double, C.c_double, C.c_int,
                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_int]),
    "tb_de_step_end": (C.c_int, [C.c_void_p, C.c_void_p]),
    "tb_de_evaluate_shard": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_double, C.c_int, C.c_int, C.c_int]),
    "tb_de_device_ptr": (C.c_void_p, [C.c_void_p, C.c_int]),
    "tb_de_get": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_size_t]),
    "tb_de_set_removed": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int]),
    "tb_de_ban_genome": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "tb_de_evaluate_testing": (C.c_int, [C.c_void_p, C.c_int, C.c_double, C.c_int, C.c_void_p]),
    "tb_marker_stats": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "tb_knockout": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_int, C.c_double, C.c_void_p,
                              C.c_void_p, C.c_void_p, C.c_void_p]),
    "tb_knockout_scan": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_int, C.c_void_p]),
    "tb_set_stream": (C.c_int, [C.c_void_p, C.c_void_p]),
    "tb_microbench": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "tb_fit_effects": (C.c_int, [C.c_void_p, C.c_int, C.c_double, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.c_void_p]),
    "tb_predict_effects": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_int, C.c_void_p]),
    "tb_reml_profile": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                  C.c_void_p]),
}

_lib = None


class TblupLibraryError(RuntimeError):
    pass


def load():
    """Load the shared library (once) and bind the prototypes.  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise TblupLibraryError(
            "%s not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or make -C tblup_b200/csrc). tblup_b200 has no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)          # AttributeError here means header and library disagree
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib

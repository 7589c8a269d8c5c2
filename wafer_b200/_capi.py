"""ctypes declarations for include/wafer_b200.h.  Loading fails loudly: there is no Python/CPU fallback."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# WAFER_B200_LIB: another build of the same library (to compare two builds in one session); never a fallback
LIB_PATH = os.environ.get("WAFER_B200_LIB") or os.path.join(_HERE, "libwafer_b200.so")

_dp = C.POINTER(C.c_double)


class Params(C.Structure):
    _fields_ = [("nx", C.c_uint64), ("ny", C.c_uint64), ("nz", C.c_uint64), ("ext", C.c_uint32),
                ("dn", C.c_double), ("dt", C.c_double), ("mass", C.c_double), ("device", C.c_int32),
                ("rank", C.c_uint32), ("world", C.c_uint32), ("nccl_id", C.POINTER(C.c_uint8)),
                ("max_lower", C.c_uint32), ("flags", C.c_uint32)]


class Observables(C.Structure):
    _fields_ = [("energy", C.c_double), ("norm2", C.c_double), ("v_infinity", C.c_double), ("r2", C.c_double)]


class Record(C.Structure):
    _fields_ = [("step", C.c_uint64), ("tau", C.c_double), ("diff", C.c_double), ("obs", Observables)]


class WriteStats(C.Structure):
    _fields_ = [("bytes", C.c_uint64), ("file_bytes", C.c_uint64), ("host_formatted", C.c_uint64)]


class LoadStats(C.Structure):
    _fields_ = [("sx", C.c_uint64), ("sy", C.c_uint64), ("sz", C.c_uint64), ("bytes_read", C.c_uint64),
                ("sites_converted", C.c_uint64), ("host_converted", C.c_uint64)]


# every symbol include/wafer_b200.h declares: name -> (restype, argtypes)
_ctx = C.c_void_p
SYMBOLS = {
    "wafer_create": (C.c_int, [C.POINTER(Params), C.POINTER(_ctx)]),
    "wafer_destroy": (C.c_int, [_ctx]),
    "wafer_last_error": (C.c_char_p, [_ctx]),
    "wafer_nccl_unique_id": (C.c_int, [C.POINTER(C.c_uint8)]),
    "wafer_slab": (C.c_int, [_ctx, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "wafer_slab_partition": (C.c_int, [C.c_uint64, C.c_uint32, C.c_uint32, C.POINTER(C.c_uint64),
                                       C.POINTER(C.c_uint64)]),
    "wafer_tb2_plan": (C.c_int, [C.c_uint32, C.c_uint32, C.c_int32, C.c_int32, C.c_uint32, C.POINTER(C.c_int32), C.c_uint64,
                                 C.POINTER(C.c_uint64)]),
    "wafer_set_potential": (C.c_int, [_ctx, _dp]),
    "wafer_get_potential": (C.c_int, [_ctx, _dp]),
    "wafer_set_pot_sub_scalar": (C.c_int, [_ctx, C.c_double]),
    "wafer_set_pot_sub_array": (C.c_int, [_ctx, _dp]),
    "wafer_set_phi": (C.c_int, [_ctx, _dp]),
    "wafer_get_phi": (C.c_int, [_ctx, _dp]),
    "wafer_slab_planes": (C.c_int, [_ctx, C.c_int32, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "wafer_set_phi_slab": (C.c_int, [_ctx, _dp]),
    "wafer_get_phi_slab": (C.c_int, [_ctx, _dp]),
    "wafer_set_phi_owned": (C.c_int, [_ctx, _dp]),
    "wafer_push_lower": (C.c_int, [_ctx, _dp]),
    "wafer_push_lower_from_phi": (C.c_int, [_ctx]),
    "wafer_get_lower": (C.c_int, [_ctx, C.c_uint32, _dp]),
    "wafer_phi_from_lower": (C.c_int, [_ctx, C.c_uint32]),
    "wafer_phi_seed_from_lower": (C.c_int, [_ctx, C.c_uint32]),
    "wafer_clear_lowers": (C.c_int, [_ctx]),
    "wafer_num_lowers": (C.c_uint32, [_ctx]),
    "wafer_generate_potential": (C.c_int, [_ctx, C.c_int32, C.c_double]),
    "wafer_generate_initial_condition": (C.c_int, [_ctx, C.c_int32]),
    "wafer_generate_gaussian": (C.c_int, [_ctx, C.c_double, C.c_uint64]),
    "wafer_symmetrise": (C.c_int, [_ctx, C.c_int32]),
    "wafer_set_phi_resampled": (C.c_int, [_ctx, _dp, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint32]),
    "wafer_set_potential_resampled": (C.c_int, [_ctx, _dp, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint32]),
    "wafer_push_lower_resampled": (C.c_int, [_ctx, _dp, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint32]),
    "wafer_write_array": (C.c_int, [_ctx, C.c_int32, C.c_int32, C.c_char_p, C.POINTER(WriteStats)]),
    "wafer_load_array": (C.c_int, [_ctx, C.c_int32, C.c_int32, C.c_char_p, C.POINTER(LoadStats)]),
    "wafer_observables_compute": (C.c_int, [_ctx, C.POINTER(Observables)]),
    "wafer_norm2": (C.c_int, [_ctx, _dp]),
    "wafer_normalise": (C.c_int, [_ctx, C.c_double]),
    "wafer_orthogonalise": (C.c_int, [_ctx, C.c_uint8]),
    "wafer_evolve": (C.c_int, [_ctx, C.c_uint8, C.c_uint64]),
    "wafer_check": (C.c_int, [_ctx, C.c_uint8, C.POINTER(Observables)]),
    "wafer_solve": (C.c_int, [_ctx, C.c_uint8, C.c_double, C.c_int64, C.c_uint64, C.c_uint64, C.POINTER(Record),
                              C.c_uint64, C.POINTER(C.c_uint64)]),
    "wafer_synchronize": (C.c_int, [_ctx]),
    "wafer_timer_begin": (C.c_int, [_ctx]),
    "wafer_timer_end": (C.c_int, [_ctx, _dp]),
    "wafer_kernel_launches": (C.c_uint64, [_ctx]),
    "wafer_host_alloc": (C.c_int, [C.POINTER(C.c_void_p), C.c_size_t]),
    "wafer_host_free": (C.c_int, [C.c_void_p]),
    "wafer_host_register": (C.c_int, [C.c_void_p, C.c_size_t]),
    "wafer_host_unregister": (C.c_int, [C.c_void_p]),
    "wafer_device_info": (C.c_int, [_ctx, C.c_char_p, C.c_size_t, C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                    C.POINTER(C.c_int32), C.POINTER(C.c_uint64)]),
    "wafer_p2p_export": (C.c_int, [_ctx, C.POINTER(C.c_uint8)]),
    "wafer_p2p_connect": (C.c_int, [_ctx, C.POINTER(C.c_uint8), C.POINTER(C.c_uint8)]),
    "wafer_selftest_division": (C.c_int, [_ctx, C.c_double, C.c_uint64, C.c_uint64, C.POINTER(C.c_uint64)]),
    "wafer_phi_checksum": (C.c_int, [_ctx, C.c_uint64, C.c_uint64, C.POINTER(C.c_uint64)]),
    "wafer_debug_halo_delay": (C.c_int, [_ctx, C.c_uint64]),
    "wafer_version": (C.c_char_p, []),
    "wafer_sweep_variant": (C.c_char_p, [_ctx]),
}

_lib = None


def load():
    """dlopen the in-tree CUDA library.  Raises (never falls back) when it is missing or incomplete."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError("%s is missing: run `make` (or __graft_entry__.build()); wafer_b200 has no CPU fallback"
                              % LIB_PATH)
        lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(lib, name)  # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib

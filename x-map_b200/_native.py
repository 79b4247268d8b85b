"""ctypes binding of libxmap_b200.so (the C ABI declared in include/xmap_b200.h).

There is no CPU fallback: if the shared library is missing or a call fails the
caller gets an exception.  Build it with ``python -c "import __graft_entry__ as
g; g.build()"`` (nvcc, sm_100a).
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("XMAP_B200_LIB") or os.path.join(_HERE, "libxmap_b200.so")

KMAX = 64
XSIM_MAX_CELLS_LG = 13    # XMAP_XSIM_MAX_CELLS_LG
METHODS = {"adjust_cosine": 0, "cosine": 1}
SELECT_LONG = 8192            # XMAP_SELECT_LONG
ABI_VERSION = 10
ROW_HDR_BYTES = 48          # XMAP_SIM_ROW_HDR_BYTES
INGEST_ID_MAX = 48          # XMAP_INGEST_ID_MAX

_p = C.c_void_p


class SimArgs(C.Structure):
    _fields_ = [
        ("csc_ptr", _p), ("csc_ent", _p), ("csc_aux", _p), ("tcsr_ent", _p),
        ("ostat", _p), ("ord", _p), ("tri_work", _p), ("ord_item", _p),
        ("dom_code", _p), ("contains", _p),
        ("n_items", C.c_int32), ("method", C.c_int32), ("num_atleast", C.c_int32),
        ("k", C.c_int32), ("r2_bits", C.c_int32), ("count_only", C.c_int32),
        ("rec_ptr", _p), ("rec_cnt", _p), ("rec", _p), ("rec_n", _p), ("bb", _p), ("row_npairs", _p),
        ("tab_idx", _p), ("tab_sim", _p), ("tab_mutu", _p), ("tab_n", _p), ("tab_len", _p),
        ("error_flag", _p), ("unit_cycles", _p),
    ]


class XsimArgs(C.Structure):
    _fields_ = [
        ("n_starts", C.c_int32), ("n_units", C.c_int32),
        ("unit_order", _p), ("unit_counter", _p), ("warps", C.c_int32), ("unit_leg_lo", _p), ("unit_leg_hi", _p),
        ("unit_g0", _p), ("unit_g1", _p), ("unit_npass", _p), ("start_unit_ptr", _p),
        ("lp_ptr", _p), ("pd_s", _p), ("pd_n", _p), ("pd_d", _p), ("pd_c", _p),
        ("rs_ptr", _p), ("rs_end", _p), ("rs_n", _p), ("rs_d", _p), ("rs_c", _p),
        ("tile_ptr", _p), ("gb", C.c_int32),
        ("cells_lg", C.c_int32), ("unit_clg", _p), ("gws", _p), ("gcells_lg", C.c_int32),
        ("top_m", C.c_int32),
        ("unit_count", _p), ("unit_combos", _p), ("unit_top_end", _p), ("unit_top_xsim", _p), ("unit_top_len", _p),
        ("out_count", _p), ("out_combos", _p), ("top_end", _p), ("top_xsim", _p), ("top_len", _p),
        ("emit_ptr", _p), ("emit_end", _p), ("emit_xsim", _p),
        ("error_flag", _p), ("unit_cycles", _p),
    ]


_SIGS = {
    "xmap_abi_version": (C.c_int, []),
    "xmap_last_error": (C.c_char_p, []),
    "xmap_layout_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int32, C.c_int32]),
    "xmap_build_layout": (C.c_int, [_p, _p, _p, C.c_int64, C.c_int32, C.c_int32,
                                    _p, _p, _p, _p, _p, _p, _p, _p, C.c_size_t, _p]),
    "xmap_row_work": (C.c_int, [_p, _p, _p, C.c_int32, _p, _p]),
    "xmap_tri_workspace_bytes": (C.c_size_t, [C.c_int64]),
    "xmap_build_tri_layout": (C.c_int, [_p, _p, _p, _p, _p, _p, _p, _p, C.c_int32, C.c_int32, C.c_int64, C.c_int32,
                                        C.c_int32, _p, _p, _p, _p, _p, C.c_size_t, _p]),
    "xmap_sim_row_cells": (C.c_int64, [C.c_int64, C.c_int32]),
    "xmap_sim_accumulate": (C.c_int, [C.POINTER(SimArgs), _p, C.c_int32, C.c_int32, C.c_int32, _p, C.c_int32, _p]),
    "xmap_sim_row_headers": (C.c_int, [C.POINTER(SimArgs), _p, C.c_int32, _p, _p, _p, _p]),
    "xmap_sim_accumulate_split": (C.c_int, [C.POINTER(SimArgs), _p, _p, _p, C.c_int32, C.c_int32, _p, _p, _p]),
    "xmap_sim_select": (C.c_int, [C.POINTER(SimArgs), _p, C.c_int32, C.c_int32, _p]),
    "xmap_segmented_copy16": (C.c_int, [_p, _p, _p, _p, _p, C.c_int32, C.c_int64, _p]),
    "xmap_segmented_copy4": (C.c_int, [_p, _p, _p, _p, _p, C.c_int32, C.c_int64, _p]),
    "xmap_xsim_smem_bytes": (C.c_int64, [C.c_int32, C.c_int32]),
    "xmap_xsim_extend": (C.c_int, [C.POINTER(XsimArgs), _p]),
    "xmap_xsim_merge": (C.c_int, [C.POINTER(XsimArgs), _p]),
    "xmap_xsim_cta_smem_bytes": (C.c_int64, [C.c_int32]),
    "xmap_xsim_extend_cta": (C.c_int, [C.POINTER(XsimArgs), _p]),
    "xmap_recsim_item_info": (C.c_int, [_p, _p, C.c_int32, _p, _p]),
    "xmap_recsim_fill_rows": (C.c_int, [_p, C.c_int32, _p, _p, C.c_int64, _p, C.c_int64, C.c_int32, C.c_int32, C.c_int64,
                                        _p, _p, _p]),
    "xmap_recsim_pairs": (C.c_int, [_p, _p, _p, _p, _p, C.c_int64, C.c_int64, C.c_int32, _p, _p, _p, _p, _p, _p]),
    "xmap_recsim_neighbors": (C.c_int, [_p, _p, _p, C.c_int32, C.c_int32, _p, _p, _p, _p]),
    "xmap_recsim_predict": (C.c_int, [_p, _p, _p, _p, _p, _p, _p, _p, C.c_int32, _p, _p, C.c_int64, C.c_double,
                                      _p, _p, _p, _p]),
    "xmap_recsim_private_neighbor": (C.c_int, [_p, _p, _p, _p, C.c_int32, C.c_int32, C.c_double, C.c_double, _p, _p, C.c_uint64,
                                               _p, _p, _p, _p, _p]),
    "xmap_clean_records": (C.c_int, [_p, _p, _p, _p, C.c_int64, C.c_int32, C.c_double, C.c_double, C.c_int32, _p, _p, _p]),
    "xmap_choose_mapping": (C.c_int, [_p, _p, _p, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                      C.c_double, C.c_int32, C.c_int32, _p, C.c_uint64, _p, _p]),
    "xmap_invert_mapping": (C.c_int, [_p, _p, C.c_int32, _p, _p]),
    "xmap_alterego_workspace_bytes": (C.c_size_t, [C.c_int64]),
    "xmap_build_alterego": (C.c_int, [_p, _p, _p, _p, C.c_int32, C.c_int64, _p,
                                      _p, _p, _p, _p, C.POINTER(C.c_int64), _p, C.c_size_t, _p]),
    "xmap_ingest_line_masks": (C.c_int, [_p, C.c_int64, _p, _p, _p]),
    "xmap_ingest_line_offsets": (C.c_int, [_p, C.c_int64, _p, _p, _p]),
    "xmap_ingest_parse": (C.c_int, [_p, _p, C.c_int64, C.c_char_p, C.c_int32, C.c_double, C.c_double, C.c_int64,
                                    _p, _p, _p, _p, _p, _p, _p, _p]),
    "xmap_ingest_rank_flags": (C.c_int, [_p, C.c_int64, C.c_int32, _p, C.c_int64, _p, _p]),
    "xmap_ingest_rank_scatter": (C.c_int, [_p, _p, _p, C.c_int64, _p, _p, _p]),
    "xmap_ingest_first": (C.c_int, [_p, _p, _p, _p, _p, C.c_int64, C.c_double, C.c_double, _p, _p, _p]),
    "xmap_ingest_item_suffix": (C.c_int, [_p, C.c_int64, _p, _p, C.c_int32, _p, _p]),
    "xmap_ingest_item_codes": (C.c_int, [_p, C.c_int64, _p, _p, C.c_int32, _p, C.c_int32, _p, _p, _p, _p, _p, _p]),
    "xmap_ingest_train_keys": (C.c_int, [_p, _p, _p, _p, _p, _p, C.c_int64, _p, _p]),
}

EXPORTED_SYMBOLS = tuple(_SIGS)

_lib = None


class NativeError(RuntimeError):
    pass


def lib():
    """Load the shared library once; raise loudly if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise NativeError(
                "%s is missing: the CUDA extension has not been built "
                "(run __graft_entry__.build()); xmap_b200 has no CPU fallback" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        if L.xmap_abi_version() != ABI_VERSION:
            raise NativeError("libxmap_b200.so ABI version mismatch")
        _lib = L
    return _lib


def check(rc, what):
    if rc != 0:
        raise NativeError("%s failed (%d): %s" % (what, rc, lib().xmap_last_error().decode()))


def ptr(t):
    """Device pointer of a torch tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()

"""ctypes binding of libcfk.so (include/cfk.h).  There is no fallback: if the CUDA
library is missing or an entry point fails, the caller gets an exception."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CFK_LIBRARY") or os.path.join(_HERE, "libcfk.so")  # override: tuning experiments only

_p = ctypes.c_void_p
_i64 = ctypes.c_int64
_i32 = ctypes.c_int32
_u32 = ctypes.c_uint32
_int = ctypes.c_int
_f64 = ctypes.c_double

# name -> (restype, argtypes); must list every symbol include/cfk.h declares
# (tests/test_abi.py cross-checks this table against the header and the built library)
SIGNATURES = {
    "cfk_abi_version": (_int, []),
    "cfk_last_error": (ctypes.c_char_p, []),
    "cfk_pair_table_bytes_per_warp": (_int, []),
    "cfk_pair_warps_per_block": (_int, []),
    "cfk_launch_count": (_i64, []),
    "cfk_table_init": (_int, [_p, _i64, _p]),
    "cfk_docfreq_count": (_int, [_p, _p, _p, _p, _i64, _int, _p, _i64, _p, _i32, _p]),
    "cfk_docfreq_plan": (_int, [_p, _p, _i64, _int, _p, _p]),
    "cfk_docfreq_count_resident": (_int, [_p, _p, _p, _p, _p, _i64, _int, _p, _i64, _p, _i32, _p]),
    "cfk_docfreq_part_target": (_int, []),
    "cfk_docfreq_part_distinct": (_int, []),
    "cfk_docfreq_emit_plan": (_int, [_p, _p, _i64, _int, _p, _p]),
    "cfk_docfreq_emit": (_int, [_p, _p, _p, _p, _p, _i64, _int, _p, _i64, _i64, _p, _p, _i32, _p]),
    "cfk_records_pack": (_int, [_p, _i64, _p, _p, _i64, _p, _p]),
    "cfk_docfreq_count_parts": (_int, [_p, _i64, _p, _p, _i64, _i32, _i64, _i32, _int, _u32, _u32, _u32, _p, _p, _p, _i64, _p,
                                       _i64, _p, _i32, _p]),
    "cfk_kmer_count_tile": (_int, []),
    "cfk_kmer_count_total": (_int, [_p, _p, _p, _p, _p, _i64, _int, _p, _i64, _p, _p]),
    "cfk_kmer_count_canonical": (_int, [_p, _p, _p, _p, _p, _i64, _int, _p, _i64, _p, _p]),
    "cfk_merge_sorted_runs": (_int, [_p, _p, _i32, _i64, _p, _p]),
    "cfk_kmer_position_keys": (_int, [_p, _i64, _int, _int, _p, _p]),
    "cfk_adjacent_gaps": (_int, [_p, _i64, _int, _p, _p]),
    "cfk_rr_max_symbols": (_int, []),
    "cfk_rr_words": (_int, [_i32]),
    "cfk_rr_filter": (_int, [_p, _p, _p, _p, _i64, _p, _p, _i32, _i32, _i32, _p, _p, _p]),
    "cfk_rr_filter_units": (_int, [_p, _p, _p, _p, _i64, _i32, _p, _p, _p, _p, _p, _p]),  # unit_m, unit_threshold: host
    "cfk_rr_long_words": (_int, [_i32]),
    "cfk_rr_filter_long": (_int, [_p, _p, _p, _p, _i64, _i32, _p, _p, _p, _p, _i32, _p, _p, _p]),  # unit_m, unit_threshold: host
    "cfk_seq_scan": (_int, [_p, _i64, _i32, _p, _i64, _p, _i64, _p]),  # host pointers
    "cfk_rr_gather": (_int, [_p, _p, _i64, _p, _i64, _p]),
    "cfk_rr_keep_sizes": (_int, [_p, _p, _p, _i64, _p, _p]),
    "cfk_rr_emit": (_int, [_p, _p, _p, _p, _i64, _i64, _p, _p]),
    "cfk_bgzf_blocks": (_int, [_p, _i64, _p, _i64, _p]),  # host pointers
    "cfk_bgzf_inflate": (_int, [_p, _p, _i64, _p, _p, _p]),
    "cfk_bam_scan": (_int, [_p, _i64, _i32, _i32, _i64, _i64, _p, _i64, _p, _p]),  # host pointers
    "cfk_rr_bam_gather": (_int, [_p, _p, _p, _i64, _p, _i64, _p]),
    "cfk_placer_best_blocks": (_int, []),
    "cfk_placer_add_read": (_int, [_p, _p, _i64, _i32, _i64, _i64, _u32, _p, _p, _i64, _p, _p, _i64, _p, _p]),
    "cfk_placer_initial_pairs": (_int, [_p, _i64, _p, _p, _i64, _p, _p]),
    "cfk_placer_update": (_int, [_p, _p, _i64, _p, _p, _p, _p, _p, _p, _i64, _p, _p, _i64, _p, _p]),
    "cfk_placer_best": (_int, [_p, _p, _i64, _p, _p, _u32, _u32, _u32, _p, _p]),
    "cfk_table_merge": (_int, [_p, _p, _p, _i64, _p, _i64, _p, _p]),
    "cfk_table_select": (_int, [_p, _i64, _u32, _u32, _u32, _i32, _i32, _p, _p, _p, _i64, _p, _p]),
    "cfk_table_lookup": (_int, [_p, _i64, _p, _i64, _p, _p, _p]),
    "cfk_table_part_count": (_int, [_p, _i64, _i32, _p, _p]),
    "cfk_table_part_scatter": (_int, [_p, _i64, _i32, _p, _p, _p, _p, _p]),
    "cfk_sort_u64": (_int, [_p, _i64, _p]),
    "cfk_index_build": (_int, [_p, _i64, _p, _p, _i64, _p, _p]),
    "cfk_cloud_build": (_int, [_p, _p, _p, _p, _i64, _int, _p, _p, _i64, _p, _i32, _p, _p, _p]),
    "cfk_index_filter_build": (_int, [_p, _i64, _i32, _p, _p]),
    "cfk_scan_scratch_elems": (_i64, [_i64]),
    "cfk_exclusive_scan": (_int, [_p, _p, _i64, _p, _p]),
    "cfk_cloud_compact": (_int, [_p, _p, _p, _i64, _p, _p]),
    "cfk_id_histogram": (_int, [_p, _p, _i64, _i64, _p, _p]),
    "cfk_cloud_filter_count": (_int, [_p, _p, _i64, _p, _i64, _i64, _p, _p]),
    "cfk_cloud_filter_write": (_int, [_p, _p, _i64, _p, _i64, _i64, _p, _p, _p]),
    "cfk_occ_fill": (_int, [_p, _p, _i64, _i64, _p, _i64, _p, _p, _p]),
    "cfk_occ_sort": (_int, [_p, _p, _i64, _p]),
    "cfk_occ_slice_histogram": (_int, [_p, _p, _i64, _i64, _i64, _p, _p]),
    "cfk_occ_slice_fill": (_int, [_p, _p, _i64, _i64, _i64, _p, _p, _p, _p]),
    "cfk_occ_last": (_int, [_p, _i64, _p, _p, _p]),
    "cfk_unit_splits": (_int, [_p, _p, _i64, _i64, _i64, _p, _p]),
    "cfk_pair_candidates": (_int, [_p, _p, _p, _p, _p, _p, _i64, _i64, _i64, _i64, _i32, _i32, _i32, _u32, _p, _i64, _p,
                                   _i32, _p]),
    "cfk_sketch_bits": (_int, []),
    "cfk_sketch_warps_per_block": (_int, []),
    "cfk_sketch_codes_elems": (_i64, [_i64, _i64]),
    "cfk_sketch_codes": (_int, [_p, _p, _i64, _p, _p, _p]),
    "cfk_pair_sketch": (_int, [_p, _p, _p, _p, _p, _p, _p, _p, _i64, _i64, _i64, _i64, _i32, _i32, _i32, _u32, _p, _i64, _p,
                               _i32, _p]),
    "cfk_pair_join": (_int, [_p, _i64, _p, _p, _p, _p, _i32, _i32, _u32, _f64, _p, _i64, _p, _p, _p]),
    "cfk_flag_indices": (_int, [_p, _i64, _p, _p, _p]),
    # native NCRF ingestion (host pointers)
    "cfk_ncrf_last_error": (ctypes.c_char_p, []),
    "cfk_ncrf_open": (_int, [ctypes.c_char_p, _i64, _i32, _i32, ctypes.POINTER(_p)]),
    "cfk_ncrf_n_records": (_i64, [_p]),
    "cfk_ncrf_n_seen": (_i64, [_p]),
    "cfk_ncrf_n_words": (_i64, [_p]),
    "cfk_ncrf_n_bases": (_i64, [_p]),
    "cfk_ncrf_n_units": (_i64, [_p]),
    "cfk_ncrf_ids_bytes": (_i64, [_p]),
    "cfk_ncrf_export": (_int, [_p, _p, _p, _p, _p, _p, _p, _p, _p, _p]),
    "cfk_ncrf_close": (None, [_p]),
    # native edge file writer (host pointers)
    "cfk_writer_last_error": (ctypes.c_char_p, []),
    "cfk_write_edges": (_int, [ctypes.c_char_p, _p, _i64, _i32, _p, _p, _p, _p, _i64, _i32]),
    "cfk_write_edges_rows": (_int, [ctypes.c_char_p, _p, _i64, _i32, _p, _i64, _i32]),
}

_lib = None


class CfkError(RuntimeError):
    pass


def load():
    """Load libcfk.so once; raises if it has not been built (python -m centroflye_b200.build)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise CfkError(f"{LIB_PATH} is missing: build it with `python -m centroflye_b200.build` "
                           "(there is no CPU fallback for the recruitment path)")
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def call(name, *args):
    """Call an int-returning entry point; non-zero status -> CfkError with cfk_last_error()."""
    lib = load()
    rc = getattr(lib, name)(*args)
    if rc != 0:
        raise CfkError(f"{name} failed ({rc}): {lib.cfk_last_error().decode(errors='replace')}")
    return rc

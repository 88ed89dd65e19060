"""ctypes binding of libsweepga_b200.so (the C ABI declared in include/sweepga_b200.h).

The library is built in-tree by __graft_entry__.build(); importing this module fails loudly when it is
missing — there is no Python or CPU fallback for any compute entry point.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libsweepga_b200.so")

u8p, u32p, u64p, f64p = C.POINTER(C.c_uint8), C.POINTER(C.c_uint32), C.POINTER(C.c_uint64), C.POINTER(C.c_double)

NO_LIMIT = (1 << 64) - 1
KEEP_ALL = (1 << 64) - 1
ONE_TO_ONE, ONE_TO_MANY, MANY_TO_MANY = 0, 1, 2
SCORE_IDENTITY, SCORE_LENGTH, SCORE_LENGTH_IDENTITY, SCORE_LOG_LENGTH_IDENTITY, SCORE_MATCHES = range(5)
DROPPED, SCAFFOLD, RESCUED, UNASSIGNED = range(4)
OK, ERR_ARG, ERR_RANGE, ERR_CUDA, ERR_OOM, ERR_IO, ERR_PARSE, ERR_UNSUPPORTED = 0, -1, -2, -3, -4, -5, -6, -7
# columns of swg_filter_batch's per-table counts
TC_STAGE1, TC_KEPT, TC_SCAFFOLD, TC_RESCUED, TC_CHAINS_KEPT, TC_COUNT = range(6)


class swg_config(C.Structure):
    _fields_ = [
        ("min_block_length", C.c_uint64), ("mapping_max_per_query", C.c_uint64), ("mapping_max_per_target", C.c_uint64),
        ("scaffold_max_per_query", C.c_uint64), ("scaffold_max_per_target", C.c_uint64), ("scaffold_gap", C.c_uint64),
        ("min_scaffold_length", C.c_uint64), ("scaffold_max_deviation", C.c_uint64),
        ("overlap_threshold", C.c_double), ("scaffold_overlap_threshold", C.c_double),
        ("min_identity", C.c_double), ("min_scaffold_identity", C.c_double),
        ("mapping_filter_mode", C.c_uint8), ("scaffold_filter_mode", C.c_uint8), ("scoring_function", C.c_uint8),
        ("keep_self", C.c_uint8), ("scaffolds_only", C.c_uint8), ("reserved", C.c_uint8 * 3),
    ]


class swg_mappings(C.Structure):
    _fields_ = [
        ("n", C.c_uint64), ("query_id", u32p), ("target_id", u32p), ("query_start", u32p), ("query_end", u32p),
        ("target_start", u32p), ("target_end", u32p), ("block_length", u32p), ("matches", u32p),
        ("identity", f64p), ("strand", u8p), ("score", f64p), ("n_seq", C.c_uint32),
        ("seq_genome_id", u32p), ("seq_genome2_id", u32p), ("query_id16", C.POINTER(C.c_uint16)), ("target_id16", C.POINTER(C.c_uint16)),
    ]


class swg_result(C.Structure):
    _fields_ = [("status", u8p), ("chain_id", u32p)]


class swg_stats(C.Structure):
    _fields_ = [
        ("n_input", C.c_uint64), ("n_stage1", C.c_uint64), ("n_after_sweep", C.c_uint64), ("n_chains", C.c_uint64),
        ("n_chains_after_mass", C.c_uint64), ("n_chains_kept", C.c_uint64), ("n_anchors", C.c_uint64),
        ("n_rescued", C.c_uint64), ("n_kept", C.c_uint64), ("score_near_ties", C.c_uint64), ("gpu_launches", C.c_uint64),
        ("ms_h2d", C.c_double), ("ms_device", C.c_double), ("ms_d2h", C.c_double),
        ("ms_sort_passes", C.c_double), ("n_sort_passes", C.c_uint64), ("n_sort_pairs", C.c_uint64),
        ("ms_tokenize", C.c_double), ("ms_write", C.c_double), ("exact_rerank", C.c_uint64), ("sort_bytes_per_pair", C.c_uint64),
        ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64), ("n_dirty_groups", C.c_uint64),
        ("ms_prefilter", C.c_double), ("prefilter_bytes_per_record", C.c_uint64), ("n_unsorted_groups", C.c_uint64),
    ]


# every symbol include/sweepga_b200.h declares: (name, restype, argtypes)
_vp = C.c_void_p
_cfgp, _mapp, _resp, _statp = C.POINTER(swg_config), C.POINTER(swg_mappings), C.POINTER(swg_result), C.POINTER(swg_stats)
_sweep_args = [_vp, C.c_uint64, u32p, u32p, u32p, u32p, f64p, C.c_uint64, C.c_double, C.c_int, u8p]
SYMBOLS = [
    ("swg_config_default", None, [_cfgp]),
    ("swg_create", _vp, [C.c_int]),
    ("swg_destroy", None, [_vp]),
    ("swg_last_error", C.c_char_p, [_vp]),
    ("swg_filter", C.c_int, [_vp, _cfgp, _mapp, _resp, _statp]),
    ("swg_filter_device", C.c_int, [_vp, _cfgp, _mapp, _resp, _statp]),
    ("swg_stream", _vp, [_vp]),
    ("swg_prefetch", C.c_int, [_vp, _mapp]),
    ("swg_prefetch_drop", None, [_vp]),
    ("swg_filter_batch", C.c_int, [_vp, _cfgp, C.c_uint64, _mapp, _resp, u64p, _statp]),
    ("swg_upload", C.c_int, [_vp, _mapp, _mapp, _resp]),
    ("swg_release", None, [_vp, _mapp, _resp]),
    ("swg_download_result", C.c_int, [_vp, C.c_uint64, _resp, _resp]),
    ("swg_last_chain_keys", C.c_int, [_vp, C.c_uint64, u32p, u32p, u64p]),
    ("swg_score_column", C.c_int, [_vp, C.c_uint64, f64p, u32p, u32p, C.c_int, f64p]),
    ("swg_chain_identity", C.c_int, [_vp, C.c_uint64, u64p, u64p, u64p, f64p]),
    ("swg_log_matches_host", C.c_int, [_vp]),
    ("swg_glibc_log_host", C.c_double, [C.c_double]),
    ("swg_plane_sweep_core", C.c_int, [_vp, C.c_uint64, u32p, u32p, f64p, C.c_uint64, C.c_double, u64p, u64p]),
    ("swg_plane_sweep_query", C.c_int, _sweep_args),
    ("swg_plane_sweep_target", C.c_int, _sweep_args),
    ("swg_plane_sweep_both", C.c_int, [_vp, C.c_uint64, u32p, u32p, u32p, u32p, f64p, C.c_uint64, C.c_uint64, C.c_double, C.c_int, u8p]),
    ("swg_parse_filter_mode_cli", C.c_int, [C.c_char_p, u8p, u64p, u64p]),
    ("swg_parse_filter_mode_lib", C.c_int, [C.c_char_p, u8p, u64p, u64p]),
    ("swg_parse_scoring", C.c_int, [C.c_char_p, u8p]),
    ("swg_parse_metric_number", C.c_int, [C.c_char_p, u64p]),
    ("swg_parse_identity_value", C.c_int, [C.c_char_p, C.c_int, C.c_double, f64p]),
    ("swg_round_nice", C.c_uint64, [C.c_uint64]),
    ("swg_clamp_scaffold_params", None, [C.c_uint64, C.c_uint64, C.c_int, C.c_uint64, C.c_int, u64p, u64p]),
    ("swg_paf_parse", _vp, [C.c_char_p, C.c_char_p, C.c_size_t]),
    ("swg_paf_free", None, [_vp]),
    ("swg_paf_n_records", C.c_uint64, [_vp]),
    ("swg_paf_n_lines", C.c_uint64, [_vp]),
    ("swg_paf_n_seq", C.c_uint32, [_vp]),
    ("swg_paf_rank", u64p, [_vp]),
    ("swg_paf_seq_name", C.c_char_p, [_vp, C.c_uint32]),
    ("swg_paf_view", C.c_int, [_vp, _mapp]),
    ("swg_paf_write", C.c_int, [_vp, C.c_char_p, u8p, u32p]),
    ("swg_parse_ani_method", C.c_int, [C.c_char_p, C.POINTER(C.c_int), f64p, C.POINTER(C.c_int)]),
    ("swg_ani_stats", C.c_int, [_vp, C.c_char_p, C.c_int, C.c_double, C.c_int, f64p, u64p]),
    ("swg_tree_filter_paf", C.c_int, [_vp, C.c_char_p, C.c_char_p, C.c_uint64, C.c_uint64, C.c_double, u64p, u64p]),
    ("swg_paf_parse_device", _vp, [_vp, C.c_char_p]),
    ("swg_filter_paf", C.c_int, [_vp, _cfgp, C.c_char_p, C.c_char_p, _statp]),
    ("swg_filter_paf_batch", C.c_int, [_vp, _cfgp, C.c_uint64, C.POINTER(C.c_char_p), C.POINTER(C.c_char_p), u64p, _statp]),
    ("swg_filter_paf_host", C.c_int, [_vp, _cfgp, C.c_char_p, C.c_char_p, _statp]),
    ("swg_filter_file", C.c_int, [_vp, _cfgp, C.c_char_p, C.c_char_p, C.c_int, _statp]),
    ("swg_aln_to_paf", C.c_int, [C.c_char_p, C.c_char_p, C.c_int]),
    ("swg_shard_plan", C.c_int, [_mapp, C.c_int, u32p, u64p]),
    ("swg_shard_plan_units", C.c_int, [C.c_uint64, u64p, C.c_int, u32p, u64p]),
    ("swg_last_chain_units", C.c_int, [_vp, C.c_uint64, u32p, u32p, u64p]),
    ("swg_renumber_chains_device", C.c_int, [_vp, C.c_uint64, C.c_void_p, C.c_uint64, u32p, C.POINTER(C.c_int64)]),
    ("swg_pack_status_device", C.c_int, [_vp, C.c_uint64, C.c_void_p, C.c_void_p]),
    ("swg_multi_create", _vp, [C.POINTER(C.c_int), C.c_int]),
    ("swg_multi_destroy", None, [_vp]),
    ("swg_multi_last_error", C.c_char_p, [_vp]),
    ("swg_multi_device_count", C.c_int, [_vp]),
    ("swg_multi_filter", C.c_int, [_vp, _cfgp, _mapp, _resp, _statp]),
    ("swg_version", C.c_char_p, []),
]


def load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: run `python __graft_entry__.py` (nvcc, sm_100a) first. "
            "sweepga_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, res, args in SYMBOLS:
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    return lib


lib = load()

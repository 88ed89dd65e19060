//! Raw bindings to `include/sweepga_b200.h` — the C ABI that replaces the body of `PafFilter::apply_filters`
//! (sweepga `src/paf_filter.rs:379-747`) and the thin callers either side of it.  Field order, types and function
//! signatures mirror the header one to one; `tests/test_ffi_crate.py` of the sweepga_b200 repository parses this file and
//! checks every struct against the header's layout (sizeof / offsetof through gcc) and every function against the
//! header's declarations, because the crate itself cannot be compiled where that repository is developed (no cargo).
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int, c_void};

pub const SWG_NO_LIMIT: u64 = u64::MAX;
pub const SWG_KEEP_ALL: u64 = u64::MAX;

pub const SWG_ONE_TO_ONE: u8 = 0;
pub const SWG_ONE_TO_MANY: u8 = 1;
pub const SWG_MANY_TO_MANY: u8 = 2;

pub const SWG_SCORE_IDENTITY: u8 = 0;
pub const SWG_SCORE_LENGTH: u8 = 1;
pub const SWG_SCORE_LENGTH_IDENTITY: u8 = 2;
pub const SWG_SCORE_LOG_LENGTH_IDENTITY: u8 = 3;
pub const SWG_SCORE_MATCHES: u8 = 4;

pub const SWG_DROPPED: u8 = 0;
pub const SWG_SCAFFOLD: u8 = 1;
pub const SWG_RESCUED: u8 = 2;
pub const SWG_UNASSIGNED: u8 = 3;

/// Columns of the per-table counts of `swg_filter_batch` (row k, column SWG_TC_*; n_tables * SWG_TC_COUNT u64, row-major).
pub const SWG_TC_STAGE1: usize = 0;
pub const SWG_TC_KEPT: usize = 1;
pub const SWG_TC_SCAFFOLD: usize = 2;
pub const SWG_TC_RESCUED: usize = 3;
pub const SWG_TC_CHAINS_KEPT: usize = 4;
pub const SWG_TC_COUNT: usize = 5;

pub const SWG_OK: c_int = 0;
pub const SWG_ERR_ARG: c_int = -1;
pub const SWG_ERR_RANGE: c_int = -2;
pub const SWG_ERR_CUDA: c_int = -3;
pub const SWG_ERR_OOM: c_int = -4;
pub const SWG_ERR_IO: c_int = -5;
pub const SWG_ERR_PARSE: c_int = -6;
pub const SWG_ERR_UNSUPPORTED: c_int = -7;

pub const SWG_ANI_ALL: c_int = 0;
pub const SWG_ANI_ORTHOGONAL: c_int = 1;
pub const SWG_ANI_NPERCENTILE: c_int = 2;
pub const SWG_NSORT_LENGTH: c_int = 0;
pub const SWG_NSORT_IDENTITY: c_int = 1;
pub const SWG_NSORT_SCORE: c_int = 2;

#[repr(C)]
#[derive(Clone, Copy, Debug)]
pub struct swg_config {
    pub min_block_length: u64,
    pub mapping_max_per_query: u64,
    pub mapping_max_per_target: u64,
    pub scaffold_max_per_query: u64,
    pub scaffold_max_per_target: u64,
    pub scaffold_gap: u64,
    pub min_scaffold_length: u64,
    pub scaffold_max_deviation: u64,
    pub overlap_threshold: f64,
    pub scaffold_overlap_threshold: f64,
    pub min_identity: f64,
    pub min_scaffold_identity: f64,
    pub mapping_filter_mode: u8,
    pub scaffold_filter_mode: u8,
    pub scoring_function: u8,
    pub keep_self: u8,
    pub scaffolds_only: u8,
    pub reserved: [u8; 3],
}

#[repr(C)]
#[derive(Clone, Copy, Debug)]
pub struct swg_mappings {
    pub n: u64,
    pub query_id: *const u32,
    pub target_id: *const u32,
    pub query_start: *const u32,
    pub query_end: *const u32,
    pub target_start: *const u32,
    pub target_end: *const u32,
    pub block_length: *const u32,
    pub matches: *const u32,
    pub identity: *const f64,
    pub strand: *const u8,
    pub score: *const f64,
    pub n_seq: u32,
    pub seq_genome_id: *const u32,
    pub seq_genome2_id: *const u32,
    pub query_id16: *const u16,
    pub target_id16: *const u16,
}

#[repr(C)]
#[derive(Clone, Copy, Debug)]
pub struct swg_result {
    pub status: *mut u8,
    pub chain_id: *mut u32,
}

#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct swg_stats {
    pub n_input: u64,
    pub n_stage1: u64,
    pub n_after_sweep: u64,
    pub n_chains: u64,
    pub n_chains_after_mass: u64,
    pub n_chains_kept: u64,
    pub n_anchors: u64,
    pub n_rescued: u64,
    pub n_kept: u64,
    pub score_near_ties: u64,
    pub gpu_launches: u64,
    pub ms_h2d: f64,
    pub ms_device: f64,
    pub ms_d2h: f64,
    pub ms_sort_passes: f64,
    pub n_sort_passes: u64,
    pub n_sort_pairs: u64,
    pub ms_tokenize: f64,
    pub ms_write: f64,
    pub exact_rerank: u64,
    pub sort_bytes_per_pair: u64,
    pub h2d_bytes: u64,
    pub d2h_bytes: u64,
    pub n_dirty_groups: u64,
    pub ms_prefilter: f64,
    pub prefilter_bytes_per_record: u64,
    pub n_unsorted_groups: u64,
}

/// Opaque context: one per GPU and per calling thread.
#[repr(C)]
pub struct swg_ctx {
    _private: [u8; 0],
}
/// Opaque multi-device handle (one context per GPU).
#[repr(C)]
pub struct swg_multi {
    _private: [u8; 0],
}
/// Opaque parsed PAF (host front end).
#[repr(C)]
pub struct swg_paf {
    _private: [u8; 0],
}

extern "C" {
    pub fn swg_config_default(cfg: *mut swg_config);
    pub fn swg_create(device: c_int) -> *mut swg_ctx;
    pub fn swg_destroy(ctx: *mut swg_ctx);
    pub fn swg_last_error(ctx: *const swg_ctx) -> *const c_char;
    pub fn swg_filter(ctx: *mut swg_ctx, cfg: *const swg_config, host_in: *const swg_mappings, host_out: *mut swg_result, stats: *mut swg_stats) -> c_int;
    pub fn swg_filter_device(ctx: *mut swg_ctx, cfg: *const swg_config, dev_in: *const swg_mappings, dev_out: *mut swg_result, stats: *mut swg_stats) -> c_int;
    pub fn swg_stream(ctx: *mut swg_ctx) -> *mut c_void;
    pub fn swg_prefetch(ctx: *mut swg_ctx, host_in: *const swg_mappings) -> c_int;
    pub fn swg_prefetch_drop(ctx: *mut swg_ctx);
    pub fn swg_filter_batch(ctx: *mut swg_ctx, cfg: *const swg_config, n_tables: u64, host_in: *const swg_mappings,
                            host_out: *mut swg_result, table_counts: *mut u64, stats: *mut swg_stats) -> c_int;
    pub fn swg_upload(ctx: *mut swg_ctx, host_in: *const swg_mappings, dev_out: *mut swg_mappings, dev_res: *mut swg_result) -> c_int;
    pub fn swg_release(ctx: *mut swg_ctx, dev: *mut swg_mappings, dev_res: *mut swg_result);
    pub fn swg_download_result(ctx: *mut swg_ctx, n: u64, dev_res: *const swg_result, host_out: *mut swg_result) -> c_int;
    pub fn swg_last_chain_keys(ctx: *mut swg_ctx, cap: u64, first_index_genome_pair: *mut u32, first_index_group: *mut u32, n_chains: *mut u64) -> c_int;
    pub fn swg_last_chain_units(ctx: *mut swg_ctx, cap: u64, unit_first_index: *mut u32, unit_first_chain: *mut u32, n_units: *mut u64) -> c_int;
    pub fn swg_renumber_chains_device(ctx: *mut swg_ctx, n: u64, chain_id_dev: *mut u32, n_units: u64, unit_first_chain: *const u32, unit_delta: *const i64) -> c_int;
    pub fn swg_pack_status_device(ctx: *mut swg_ctx, n: u64, status_dev: *const u8, packed_dev: *mut u32) -> c_int;
    pub fn swg_multi_create(devices: *const c_int, n_devices: c_int) -> *mut swg_multi;
    pub fn swg_multi_destroy(m: *mut swg_multi);
    pub fn swg_multi_last_error(m: *const swg_multi) -> *const c_char;
    pub fn swg_multi_device_count(m: *const swg_multi) -> c_int;
    pub fn swg_multi_filter(m: *mut swg_multi, cfg: *const swg_config, host_in: *const swg_mappings, host_out: *mut swg_result, stats: *mut swg_stats) -> c_int;
    pub fn swg_plane_sweep_query(ctx: *mut swg_ctx, n: u64, qs: *const u32, qe: *const u32, ts: *const u32, te: *const u32, identity: *const f64, n_keep: u64, overlap_threshold: f64, scoring: c_int, keep: *mut u8) -> c_int;
    pub fn swg_plane_sweep_target(ctx: *mut swg_ctx, n: u64, qs: *const u32, qe: *const u32, ts: *const u32, te: *const u32, identity: *const f64, n_keep: u64, overlap_threshold: f64, scoring: c_int, keep: *mut u8) -> c_int;
    pub fn swg_plane_sweep_both(ctx: *mut swg_ctx, n: u64, qs: *const u32, qe: *const u32, ts: *const u32, te: *const u32, identity: *const f64, n_keep_query: u64, n_keep_target: u64, overlap_threshold: f64, scoring: c_int, keep: *mut u8) -> c_int;
    pub fn swg_plane_sweep_core(ctx: *mut swg_ctx, n: u64, begin: *const u32, end: *const u32, score: *const f64, max_to_keep: u64, overlap_threshold: f64, out_idx: *mut u64, n_out: *mut u64) -> c_int;
    pub fn swg_score_column(ctx: *mut swg_ctx, n: u64, identity: *const f64, query_start: *const u32, query_end: *const u32, scoring: c_int, score_out: *mut f64) -> c_int;
    pub fn swg_chain_identity(ctx: *mut swg_ctx, n: u64, total_length: *const u64, sum_block: *const u64, sum_matches: *const u64, weighted_identity_out: *mut f64) -> c_int;
    pub fn swg_log_matches_host(ctx: *const swg_ctx) -> c_int;
    pub fn swg_glibc_log_host(x: f64) -> f64;
    pub fn swg_parse_filter_mode_cli(s: *const c_char, mode: *mut u8, per_query: *mut u64, per_target: *mut u64) -> c_int;
    pub fn swg_parse_filter_mode_lib(s: *const c_char, mode: *mut u8, per_query: *mut u64, per_target: *mut u64) -> c_int;
    pub fn swg_parse_scoring(s: *const c_char, scoring: *mut u8) -> c_int;
    pub fn swg_parse_metric_number(s: *const c_char, out: *mut u64) -> c_int;
    pub fn swg_parse_identity_value(s: *const c_char, has_ani: c_int, ani_percentile: f64, out: *mut f64) -> c_int;
    pub fn swg_parse_ani_method(s: *const c_char, method: *mut c_int, percentile: *mut f64, sort: *mut c_int) -> c_int;
    pub fn swg_ani_stats(ctx: *mut swg_ctx, paf_path: *const c_char, method: c_int, percentile: f64, sort: c_int, ani50: *mut f64, n_pairs: *mut u64) -> c_int;
    pub fn swg_tree_filter_paf(ctx: *mut swg_ctx, in_path: *const c_char, out_path: *const c_char, k_nearest: u64, k_farthest: u64, random_fraction: f64, n_kept: *mut u64, n_pairs_selected: *mut u64) -> c_int;
    pub fn swg_round_nice(v: u64) -> u64;
    pub fn swg_clamp_scaffold_params(user_jump: u64, user_mass: u64, has_avg: c_int, avg_seq_len: u64, adaptive: c_int, jump_out: *mut u64, mass_out: *mut u64);
    pub fn swg_paf_parse(path: *const c_char, err: *mut c_char, err_len: usize) -> *mut swg_paf;
    pub fn swg_paf_free(p: *mut swg_paf);
    pub fn swg_paf_n_records(p: *const swg_paf) -> u64;
    pub fn swg_paf_n_lines(p: *const swg_paf) -> u64;
    pub fn swg_paf_n_seq(p: *const swg_paf) -> u32;
    pub fn swg_paf_rank(p: *const swg_paf) -> *const u64;
    pub fn swg_paf_seq_name(p: *const swg_paf, id: u32) -> *const c_char;
    pub fn swg_paf_view(p: *const swg_paf, out: *mut swg_mappings) -> c_int;
    pub fn swg_paf_write(p: *const swg_paf, out_path: *const c_char, status: *const u8, chain_id: *const u32) -> c_int;
    pub fn swg_paf_parse_device(ctx: *mut swg_ctx, path: *const c_char) -> *mut swg_paf;
    pub fn swg_filter_paf(ctx: *mut swg_ctx, cfg: *const swg_config, in_path: *const c_char, out_path: *const c_char, stats: *mut swg_stats) -> c_int;
    /// `PafFilter::filter_paf` over many independent PAF files in one call (`file_counts`: `n_files` rows of `SWG_TC_COUNT`, may be null).
    pub fn swg_filter_paf_batch(ctx: *mut swg_ctx, cfg: *const swg_config, n_files: u64, in_paths: *const *const c_char,
                                out_paths: *const *const c_char, file_counts: *mut u64, stats: *mut swg_stats) -> c_int;
    pub fn swg_filter_paf_host(ctx: *mut swg_ctx, cfg: *const swg_config, in_path: *const c_char, out_path: *const c_char, stats: *mut swg_stats) -> c_int;
    pub fn swg_filter_file(ctx: *mut swg_ctx, cfg: *const swg_config, in_path: *const c_char, out_path: *const c_char, keep_self: c_int, stats: *mut swg_stats) -> c_int;
    pub fn swg_aln_to_paf(aln_path: *const c_char, paf_path: *const c_char, threads: c_int) -> c_int;
    pub fn swg_shard_plan(host_in: *const swg_mappings, n_shards: c_int, shard_of: *mut u32, shard_sizes: *mut u64) -> c_int;
    pub fn swg_shard_plan_units(n_units: u64, unit_sizes: *const u64, n_shards: c_int, shard_of_unit: *mut u32, shard_sizes: *mut u64) -> c_int;
    pub fn swg_version() -> *const c_char;
}

/*
 * sweepga_b200.h — C ABI of the B200-native sweepga mapping filter.
 *
 * Drop-in boundary for ONE path of pangenome/sweepga: the body of
 *   PafFilter::apply_filters            (reference src/paf_filter.rs:379-747)
 * and the thin callers either side of it
 *   PafFilter::filter_paf               (src/paf_filter.rs:278-289)
 *   unified_filter::filter_file         (src/unified_filter.rs:280-347, PAF side)
 *   library_api::apply_paf_filter       (src/library_api.rs:267-281)
 *   plane_sweep_exact::plane_sweep_*    (src/plane_sweep_exact.rs:268-461)
 *   plane_sweep_core::plane_sweep       (src/plane_sweep_core.rs:80-149)
 *   CLI / library flag parsers          (src/main.rs:244-293, src/library_api.rs:31-63,
 *                                        src/cli.rs:26-130, src/pansn.rs:176-225)
 *
 * Plain pointers and sizes only; no torch / CUDA types in any signature.
 * All compute entry points run hand-written sm_100a kernels; there is NO CPU
 * fallback: every compute call fails with SWG_ERR_CUDA when no device is usable.
 *
 * The reference-side binding (Rust `extern "C"` block + build.rs) a maintainer
 * would add is shown in INTEGRATION.md.
 */
#ifndef SWEEPGA_B200_H
#define SWEEPGA_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- enums (values are part of the ABI) -------------------------------- */

/* FilterMode, reference src/filter_types.rs:17-22 */
enum { SWG_ONE_TO_ONE = 0, SWG_ONE_TO_MANY = 1, SWG_MANY_TO_MANY = 2 };

/* ScoringFunction, reference src/filter_types.rs:8-14 */
enum {
    SWG_SCORE_IDENTITY = 0,
    SWG_SCORE_LENGTH = 1,
    SWG_SCORE_LENGTH_IDENTITY = 2,
    SWG_SCORE_LOG_LENGTH_IDENTITY = 3,
    SWG_SCORE_MATCHES = 4
};

/* ChainStatus (reference src/mapping.rs:82-86) + "not in the result map" */
enum { SWG_DROPPED = 0, SWG_SCAFFOLD = 1, SWG_RESCUED = 2, SWG_UNASSIGNED = 3 };

/* return codes */
enum {
    SWG_OK = 0,
    SWG_ERR_ARG = -1,     /* NULL pointer / bad enum / bad size                          */
    SWG_ERR_RANGE = -2,   /* coordinate does not fit the u32 SoA, end < start, id >= n_seq */
    SWG_ERR_CUDA = -3,    /* no usable device / CUDA runtime error (no CPU fallback)     */
    SWG_ERR_OOM = -4,     /* device or pinned-host allocation failed                     */
    SWG_ERR_IO = -5,      /* PAF front end: cannot open / read / write                   */
    SWG_ERR_PARSE = -6,   /* flag parsers: the reference would return Err / exit         */
    SWG_ERR_UNSUPPORTED = -7 /* .1aln container without a converter (fastga-rs / ALNtoPAF)  */
};

#define SWG_NO_LIMIT (~(uint64_t)0)         /* Option<usize>::None (Some(0) stays representable) */
#define SWG_KEEP_ALL (~(uint64_t)0)         /* usize::MAX for the primitive sweeps        */

/* ---- FilterConfig (live fields only), reference src/paf_filter.rs:18-49 - */
typedef struct swg_config {
    uint64_t min_block_length;        /* --min-aln-length                                 */
    uint64_t mapping_max_per_query;   /* SWG_NO_LIMIT = None                              */
    uint64_t mapping_max_per_target;  /* SWG_NO_LIMIT = None                              */
    uint64_t scaffold_max_per_query;  /* SWG_NO_LIMIT = None                              */
    uint64_t scaffold_max_per_target; /* SWG_NO_LIMIT = None                              */
    uint64_t scaffold_gap;            /* --scaffold-jump; 0 disables scaffolding          */
    uint64_t min_scaffold_length;     /* --scaffold-mass (compared with the query SPAN)   */
    uint64_t scaffold_max_deviation;  /* --scaffold-dist; 0 = no rescue                   */
    double overlap_threshold;         /* --overlap                                        */
    double scaffold_overlap_threshold;/* --scaffold-overlap                               */
    double min_identity;              /* --min-aln-identity                               */
    double min_scaffold_identity;     /* --min-scaffold-identity                          */
    uint8_t mapping_filter_mode;      /* SWG_ONE_TO_ONE ...                               */
    uint8_t scaffold_filter_mode;
    uint8_t scoring_function;         /* SWG_SCORE_*                                      */
    uint8_t keep_self;                /* PafFilter::with_keep_self                        */
    uint8_t scaffolds_only;           /* PafFilter::with_scaffolds_only                   */
    uint8_t reserved[3];
} swg_config;

/* Defaults of the CLI (reference src/cli.rs:204-276): many:many, overlap 0.95,
 * log-length-ani, jump 50k, mass 10k, scaffold many:many, scaffold-overlap 0.5, dist 0. */
void swg_config_default(swg_config *cfg);

/* ---- compact mapping table (SoA), replaces Vec<RecordMeta> -------------- *
 * Element i is the i-th RecordMeta of the Vec handed to apply_filters (the
 * reference orders everything by Vec position; `rank` is only a map key, so the
 * caller keeps the index -> rank table).  Sequence names are interned by the
 * caller into ONE table shared by queries and targets (query_id == target_id
 * <=> same name, the --self test of src/paf_filter.rs:386).  Per sequence the
 * caller supplies the id of its genome prefix under the two prefix rules of the
 * reference:
 *   seq_genome_id   P  = name up to and including the LAST '#', else the name
 *                        (src/paf_filter.rs:1022-1030)
 *   seq_genome2_id  P2 = "f0#f1#" if the name has >= 2 '#'-separated fields,
 *                        else the name (src/plane_sweep_scaffold.rs:13-22)
 * Ids need not be first-appearance ordered; equality is all that is used.
 * Coordinates are u32 (checked by the marshaller; larger -> SWG_ERR_RANGE).    */
typedef struct swg_mappings {
    uint64_t n;
    const uint32_t *query_id;
    const uint32_t *target_id;
    const uint32_t *query_start;
    const uint32_t *query_end;
    const uint32_t *target_start;
    const uint32_t *target_end;
    const uint32_t *block_length;
    const uint32_t *matches;
    const double *identity;       /* may be NULL: identity = matches / max(block_length, 1), the parser's value for a
                                     record without dv:f: / cg:Z: tags (paf_filter.rs:322), derived on the device
                                     (same IEEE division, same bits) — 8 B per record less to upload */
    const uint8_t *strand;        /* '+' is forward; any other byte is reverse (paf_filter.rs:311) */
    const double *score;          /* optional (may be NULL): caller-computed plane-sweep score,
                                     used instead of the device-computed one (glibc-log exactness) */
    uint32_t n_seq;
    const uint32_t *seq_genome_id;
    const uint32_t *seq_genome2_id;
    /* Optional 16-bit id columns, read when query_id and target_id are both NULL and n_seq <= 65536 (HOST tables only:
     * swg_filter / swg_upload widen them on the device; swg_filter_device takes 32-bit ids): 2 B instead of 4 B per id. */
    const uint16_t *query_id16;
    const uint16_t *target_id16;
} swg_mappings;

/* Result, replaces HashMap<rank, RecordMeta{chain_id, chain_status}>.
 * status[i] = SWG_DROPPED when the record is absent from the reference's map.
 * chain_id[i] = k for "chain_k" (1-based), 0 for None.                           */
typedef struct swg_result {
    uint8_t *status;
    uint32_t *chain_id;
} swg_result;

typedef struct swg_stats {
    uint64_t n_input;
    uint64_t n_stage1;            /* after length/self/identity retain (paf_filter.rs:384-388) */
    uint64_t n_after_sweep;       /* after apply_plane_sweep_to_mappings                       */
    uint64_t n_chains;            /* merge_mappings_into_chains                                */
    uint64_t n_chains_after_mass; /* length/identity chain filter (paf_filter.rs:449-455)      */
    uint64_t n_chains_kept;       /* after the scaffold plane sweep                            */
    uint64_t n_anchors;           /* members of kept chains + captured inversions              */
    uint64_t n_rescued;
    uint64_t n_kept;              /* records with status != SWG_DROPPED                        */
    uint64_t score_near_ties;     /* score pairs within 2 ulp compared by a sweep (see DESIGN) */
    uint64_t gpu_launches;        /* kernels launched by this call                             */
    double ms_h2d, ms_device, ms_d2h; /* CUDA-event times of the three phases of swg_filter    */
    double ms_sort_passes;        /* CUDA-event time of the one-sweep passes of the record sort  */
    uint64_t n_sort_passes;       /* ... how many passes that was                               */
    uint64_t n_sort_pairs;        /* ... over how many (key,payload) pairs                      */
    double ms_tokenize;           /* swg_filter_paf: newline scan + parse + name interning on the device */
    double ms_write;              /* swg_filter_paf: output assembly on the device + download + write()  */
    uint64_t exact_rerank;        /* 1: the call was redone with every logarithm taken from the HOST libm (near ties
                                     on a host whose log() differs from the device's port, or SWG_EXACT_SCORES=always) */
    uint64_t sort_bytes_per_pair; /* bytes one timed sort pass moves per pair (24: key+payload pairs, 16: packed words) */
    uint64_t h2d_bytes, d2h_bytes;/* swg_filter: bytes copied host->device / device->host by this call        */
    uint64_t n_dirty_groups;      /* (query,target,strand) groups in which some mapping was claimed as successor twice:
                                     chained by the sequential walk instead of the one-pass claims (diagnostic)       */
    double ms_prefilter;          /* CUDA-event time of k_prefilter (stage-1 retain + sort keys), the largest kernel of a default call */
    uint64_t prefilter_bytes_per_record; /* ... and the bytes it reads + writes per input record (algorithmic)              */
    uint64_t n_unsorted_groups;   /* record sort by groups: groups of three or more records that were not in (query_start, index)
                                     order after the scatter and went through an ordering kernel (diagnostic)            */
} swg_stats;

typedef struct swg_ctx swg_ctx;

/* One context per GPU (one process per GPU in the multi-GPU driver).  Owns a
 * stream, pinned staging and grow-only HBM scratch.  Not thread-safe.
 * Returns NULL when the device cannot be initialised; the reason is then
 * available from swg_last_error(NULL).                                         */
swg_ctx *swg_create(int device);
void swg_destroy(swg_ctx *ctx);
const char *swg_last_error(const swg_ctx *ctx);

/* apply_filters with HOST buffers: H2D + filter + D2H (src/paf_filter.rs:379-747). */
int swg_filter(swg_ctx *ctx, const swg_config *cfg, const swg_mappings *host_in,
               swg_result *host_out, swg_stats *stats);

/* Same with DEVICE-resident SoA in and device-resident result out (no copies);
 * runs on the context's stream and returns after it has drained.               */
int swg_filter_device(swg_ctx *ctx, const swg_config *cfg, const swg_mappings *dev_in,
                      swg_result *dev_out, swg_stats *stats);

/* Raw stream handle (cudaStream_t) the context launches on — for event timing. */
void *swg_stream(swg_ctx *ctx);

/* Streaming hint for a caller that filters many tables back to back (one PAF per sample, per chromosome, per batch):
 * swg_prefetch() starts the host->device copy of `host_in` on the copy engine and returns at once; a later
 * swg_filter() called with a table of the SAME n and column pointers finds it on the device (oldest first) and skips its
 * own upload, so the upload of table k+1 overlaps the kernels and the result download of table k.  Up to two prefetched
 * tables per context; the host columns must stay valid and unchanged until the swg_filter call that consumes them
 * returns.  Pinned host memory overlaps; pageable memory is staged at once (no overlap).  swg_filter on any other
 * table uploads as usual.  swg_prefetch_drop() forgets the outstanding prefetches.                                      */
int swg_prefetch(swg_ctx *ctx, const swg_mappings *host_in);
void swg_prefetch_drop(swg_ctx *ctx);

/* Many independent tables in one call (one PAF per sample, per chromosome, per batch): host_out[k] receives byte for byte
 * what swg_filter writes for host_in[k] alone, chain numbers starting at chain_1 in every table, whatever else shares the
 * batch.  The tables travel as one union (ids made disjoint per table) through one run of the pipeline: one upload, one
 * kernel chain and one download instead of K, so a loop of small tables stops paying the per-call floor.  Every table may
 * use 16- or 32-bit ids and may lack `identity`; `score` is given for every table or for none (else SWG_ERR_ARG).  Tables
 * with n == 0 contribute nothing, n_tables == 0 is SWG_OK.  A NULL column (swg_last_error names the table), or more than
 * 0x7FFFFFF0 records or 2^31 sequences in all: SWG_ERR_ARG; a range error in any table fails the whole call
 * (SWG_ERR_RANGE).  table_counts (may be NULL): n_tables rows of SWG_TC_COUNT u64, row-major: records that pass the
 * stage-1 retain, records kept (status != SWG_DROPPED), SWG_SCAFFOLD, SWG_RESCUED, and the table's largest chain
 * number.  stats (may be NULL) describes the whole call (the union's stage counts, launches, phase times).  Outstanding
 * prefetches stay outstanding; afterwards the last-call chain queries report no chains.                               */
enum { SWG_TC_STAGE1 = 0, SWG_TC_KEPT = 1, SWG_TC_SCAFFOLD = 2, SWG_TC_RESCUED = 3, SWG_TC_CHAINS_KEPT = 4, SWG_TC_COUNT = 5 };
int swg_filter_batch(swg_ctx *ctx, const swg_config *cfg, uint64_t n_tables, const swg_mappings *host_in,
                     swg_result *host_out, uint64_t *table_counts, swg_stats *stats);

/* Upload a host table once / free it; lets a caller time swg_filter_device on
 * resident data without touching CUDA itself.                                   */
int swg_upload(swg_ctx *ctx, const swg_mappings *host_in, swg_mappings *dev_out, swg_result *dev_res);
void swg_release(swg_ctx *ctx, swg_mappings *dev, swg_result *dev_res);
int swg_download_result(swg_ctx *ctx, uint64_t n, const swg_result *dev_res, swg_result *host_out);

/* Order keys of the chains kept by the LAST swg_filter / swg_filter_device call on this context, for merging the
 * chain numbering of genome-pair shards filtered on different GPUs: entry k-1 describes chain_k by the input index
 * of the first stage-1 record of its genome pair (A) and of the first kept record of its (query,target,strand) group
 * (B), both taken from the FIRST filtered chain of the chain's genome-pair group (SURVEY.md Appendix B, order O3).
 * Sorting all shards' chains by (global index of A, global index of B, shard-local k) reproduces the single-GPU
 * numbering.  cap = capacity of the two arrays; *n_chains receives the count.                                  */
int swg_last_chain_keys(swg_ctx *ctx, uint64_t cap, uint32_t *first_index_genome_pair, uint32_t *first_index_group,
                        uint64_t *n_chains);

/* Merging the chain numbering of shards needs less than the per-chain keys above: the kept chains of one genome-pair unit
 * are numbered consecutively both on one GPU and in the merged numbering.  swg_last_chain_units reports, for the last
 * call, the runs of chains that share a unit: the input index A of the unit's first stage-1 record and the (1-based) local
 * number of the run's first chain, in chain order; *n_units receives the count (cap = 0: only the count).  The driver sorts
 * all shards' runs by the GLOBAL index of A, takes the exclusive prefix sum of the run lengths and hands every shard its
 * own runs' offsets: swg_renumber_chains_device adds unit_delta[r] to the chain number of every record whose chain belongs
 * to run r (chain_id_dev: DEVICE array of n entries; the run arrays: HOST).  swg_pack_status_device packs status bytes
 * into 2 bits per record (16 per u32, record i in bits 2*(i mod 16)) for the keep-bitmap gather; both arrays on the DEVICE. */
int swg_last_chain_units(swg_ctx *ctx, uint64_t cap, uint32_t *unit_first_index, uint32_t *unit_first_chain,
                         uint64_t *n_units);
int swg_renumber_chains_device(swg_ctx *ctx, uint64_t n, uint32_t *chain_id_dev, uint64_t n_units,
                               const uint32_t *unit_first_chain, const int64_t *unit_delta);
int swg_pack_status_device(swg_ctx *ctx, uint64_t n, const uint8_t *status_dev, uint32_t *packed_dev);

/* ---- primitives: plane_sweep_exact.rs:268-461 --------------------------- *
 * keep[i] = 1 iff local index i is in the Vec<usize> the reference returns.
 * n_keep = SWG_KEEP_ALL for usize::MAX.  HOST buffers.                          */
int swg_plane_sweep_query(swg_ctx *ctx, uint64_t n, const uint32_t *qs, const uint32_t *qe,
                          const uint32_t *ts, const uint32_t *te, const double *identity,
                          uint64_t n_keep, double overlap_threshold, int scoring, uint8_t *keep);
int swg_plane_sweep_target(swg_ctx *ctx, uint64_t n, const uint32_t *qs, const uint32_t *qe,
                           const uint32_t *ts, const uint32_t *te, const double *identity,
                           uint64_t n_keep, double overlap_threshold, int scoring, uint8_t *keep);
int swg_plane_sweep_both(swg_ctx *ctx, uint64_t n, const uint32_t *qs, const uint32_t *qe,
                         const uint32_t *ts, const uint32_t *te, const double *identity,
                         uint64_t n_keep_query, uint64_t n_keep_target, double overlap_threshold,
                         int scoring, uint8_t *keep);

/* plane_sweep_core::plane_sweep (src/plane_sweep_core.rs:80-149), the secondary Interval API (different semantics:
 * the n best are marked after every Begin event; greedy overlap pass in score order).  out_idx receives the kept
 * indices in the order the reference returns them (ascending, or score-descending after the overlap pass);
 * capacity n.  Events with equal (position, type) are taken in index order (the reference's sort_unstable leaves
 * that order unspecified).                                                                                     */
int swg_plane_sweep_core(swg_ctx *ctx, uint64_t n, const uint32_t *begin, const uint32_t *end, const double *score,
                         uint64_t max_to_keep, double overlap_threshold, uint64_t *out_idx, uint64_t *n_out);

/* ---- verification: the f64 expressions of the path, evaluated on the device ----------------------------------- *
 * The plane sweeps rank by score_with_function (src/plane_sweep_exact.rs:29-86: identity * ln(query span) by default)
 * and the chain filter compares weighted_identity = sum_matches / (sum_block + max(ln(gap), 0)) with a threshold
 * (src/paf_filter.rs:896-913).  The device computes ln() with a port of glibc's log (csrc/glibc_log.cuh) so that these
 * values carry the bits of the host's f64::ln; these entry points let a caller (and tests/test_scores_gpu.py) check that
 * on any argument set.  HOST buffers in and out.                                                                   */
int swg_score_column(swg_ctx *ctx, uint64_t n, const double *identity, const uint32_t *query_start,
                     const uint32_t *query_end, int scoring, double *score_out);
int swg_chain_identity(swg_ctx *ctx, uint64_t n, const uint64_t *total_length, const uint64_t *sum_block,
                       const uint64_t *sum_matches, double *weighted_identity_out);
/* 1 when swg_create found the device's ln() equal to the host libm's log() on its probe set (65 536 integer arguments),
 * 0 when not: near ties seen by a sweep then make swg_filter redo the call with host-computed logarithms
 * (swg_stats.exact_rerank; SWG_EXACT_SCORES=always|never overrides).                                               */
int swg_log_matches_host(const swg_ctx *ctx);
/* The port itself evaluated on the host (same operations, fma() from libm): lets a CPU-only test compare it with log(). */
double swg_glibc_log_host(double x);

/* ---- host-side mirrors of the flag parsers ------------------------------ */
/* src/main.rs:244-293 (CLI grammar).  *mode, *per_query, *per_target (SWG_NO_LIMIT = None). */
int swg_parse_filter_mode_cli(const char *s, uint8_t *mode, uint64_t *per_query, uint64_t *per_target);
/* src/library_api.rs:31-63 (library grammar; differs on "many:1"-style inputs).  */
int swg_parse_filter_mode_lib(const char *s, uint8_t *mode, uint64_t *per_query, uint64_t *per_target);
/* src/main.rs:3485-3492 */
int swg_parse_scoring(const char *s, uint8_t *scoring);
/* src/cli.rs:26-61 */
int swg_parse_metric_number(const char *s, uint64_t *out);
/* src/cli.rs:76-130; has_ani = 0 => ani_percentile None */
int swg_parse_identity_value(const char *s, int has_ani, double ani_percentile, double *out);
/* ---- ANI pre-pass (`--min-identity aniN`): the caller immediately before the filter ---- */
enum { SWG_ANI_ALL = 0, SWG_ANI_ORTHOGONAL = 1, SWG_ANI_NPERCENTILE = 2 };  /* AniMethod, src/main.rs:174-178 */
enum { SWG_NSORT_LENGTH = 0, SWG_NSORT_IDENTITY = 1, SWG_NSORT_SCORE = 2 }; /* NSort, src/main.rs:182-186      */
/* parse_ani_method, src/main.rs:296-331 ("all", "orthogonal" | "1:1", "nX[-length|-identity|-score]").
 * SWG_ERR_PARSE <=> None (the CLI then falls back to n50-identity, src/main.rs:3579).            */
int swg_parse_ani_method(const char *s, int *method, double *percentile, int *sort);
/* calculate_ani_stats / calculate_ani_n_percentile, src/main.rs:334-688: the median over genome pairs of
 * sum(matches) / sum(block length) over the inter-genome alignments of a PAF — all of them, the survivors of the 1:1
 * filter (ORTHOGONAL; runs swg_filter_paf into a temp file first), or the best ones in a stable descending sort
 * until their block lengths cover `percentile` % of the genome size.  The text is tokenised on the GPU and every
 * pair's f64 sums are accumulated there in the reference's order, so *ani50 is the reference's value bit for bit
 * (NSORT_SCORE: up to ties within 1 ulp of log).  SWG_ERR_RANGE when the reference would panic on a NaN. */
int swg_ani_stats(swg_ctx *ctx, const char *paf_path, int method, double percentile, int sort, double *ani50,
                  uint64_t *n_pairs);

/* apply_tree_filter_to_paf, src/tree_filter.rs:205-283 (`--sparsify tree:k[,f[,r]]` on an existing PAF): per genome
 * pair (extract_genome_prefix, :15-25) identity = sum(matches) / sum(block length); every genome keeps its k_nearest
 * and k_farthest neighbours, plus the pairs whose SipHash-1-3 is below random_fraction * 2^64 (select_tree_pairs,
 * :84-164); the lines of the selected pairs are written verbatim, in input order.  Tokenising, the per-pair integer
 * sums and the output assembly run on the GPU; the pair selection (thousands of pairs) on the host.  Ties in identity
 * go by neighbour name (the reference leaves them to HashMap iteration order). */
int swg_tree_filter_paf(swg_ctx *ctx, const char *in_path, const char *out_path, uint64_t k_nearest, uint64_t k_farthest,
                        double random_fraction, uint64_t *n_kept, uint64_t *n_pairs_selected);

/* src/pansn.rs:176-191, 207-225; has_avg = 0 => avg_seq_len None */
uint64_t swg_round_nice(uint64_t v);
void swg_clamp_scaffold_params(uint64_t user_jump, uint64_t user_mass, int has_avg, uint64_t avg_seq_len,
                               int adaptive, uint64_t *jump_out, uint64_t *mass_out);

/* ---- PAF front end (host parse -> SoA -> GPU filter -> tagged write) ----- */
typedef struct swg_paf swg_paf;
/* extract_metadata, src/paf_filter.rs:292-376 (+ parse_cigar_counts src/paf.rs:32-64). */
swg_paf *swg_paf_parse(const char *path, char *err, size_t err_len);
void swg_paf_free(swg_paf *p);
uint64_t swg_paf_n_records(const swg_paf *p);
uint64_t swg_paf_n_lines(const swg_paf *p);
uint32_t swg_paf_n_seq(const swg_paf *p);
const uint64_t *swg_paf_rank(const swg_paf *p);            /* line number of record i          */
const char *swg_paf_seq_name(const swg_paf *p, uint32_t id);
int swg_paf_view(const swg_paf *p, swg_mappings *out);     /* borrow the SoA (valid until free) */
/* write_filtered_output, src/paf_filter.rs:1689-1726 */
int swg_paf_write(const swg_paf *p, const char *out_path, const uint8_t *status, const uint32_t *chain_id);

/* extract_metadata on the device: the text is copied to HBM once and tokenised there (newline scan, field split,
 * integer / dv:f: parse, cg:Z: '=' count, name interning in first-appearance order).  Returns the same table as
 * swg_paf_parse; lines outside the plain grammar are patched by the host's line parser, and an input the device
 * declines (> 64 GiB, 64-bit name-hash collision) goes through swg_paf_parse.  NULL + swg_last_error on failure. */
swg_paf *swg_paf_parse_device(swg_ctx *ctx, const char *path);

/* PafFilter::filter_paf (src/paf_filter.rs:278-289): tokenise on the device, filter, assemble the tagged output on
 * the device (write_filtered_output, src/paf_filter.rs:1689-1726), one download, write().  stats: ms_h2d = text
 * upload, ms_tokenize, ms_device = the filter, ms_write.  SWG_PAF_FRONTEND=host selects swg_filter_paf_host. */
int swg_filter_paf(swg_ctx *ctx, const swg_config *cfg, const char *in_path, const char *out_path,
                   swg_stats *stats);
/* PafFilter::filter_paf over many independent PAF files in one call: out_paths[k] receives byte for byte what
 * swg_filter_paf(ctx, cfg, in_paths[k], out_paths[k], NULL) writes, chain numbers from chain_1 in every file, whatever else
 * shares the call.  Consecutive files travel as one union through the device front end, the filter and the writer (one
 * upload, one kernel chain, one assembled output for the group), so a loop of small files stops paying the per-call floor.
 * Files are independent tables: a sequence name that appears in two files is two sequences, and keep_self, the genome
 * prefix rules and chain numbering work per file.  Inputs are opened as swg_filter_paf opens them (plain, .gz, .bgz); every
 * out_paths[k] is created or truncated, also for an empty input.  A group stays below the limits of one file (2^31 lines,
 * 64 GiB of text), the device memory free at the start of the call and the open-file limit; SWG_PAF_BATCH_BYTES=<n> caps
 * a group's text.  A file that alone exceeds a limit is filtered as swg_filter_paf filters it; a group the device declines
 * (name-hash collision, a line over 256 MiB, too many names), and every group under SWG_PAF_FRONTEND=host, runs
 * swg_paf_parse, swg_filter_batch and swg_paf_write.  Results do not depend on the grouping.
 * file_counts (may be NULL): n_files rows of SWG_TC_COUNT u64 in the layout of swg_filter_batch's table_counts.  stats (may be
 * NULL) describes the whole call: summed stage counts, gpu_launches, ms_h2d (text upload), ms_tokenize, ms_device, ms_write.
 * n_files == 0: SWG_OK.  A NULL array or entry, or two equal out_paths strings: SWG_ERR_ARG.  An input that cannot be
 * opened: SWG_ERR_IO before any output is created; an output that cannot be created: SWG_ERR_IO; a range error in any file
 * fails the call with SWG_ERR_RANGE.  swg_last_error names the file.  On an error, the outputs of groups that already
 * finished may exist.  The context stays usable; outstanding prefetches stay outstanding; afterwards the last-call chain
 * queries report no chains.  */
int swg_filter_paf_batch(swg_ctx *ctx, const swg_config *cfg, uint64_t n_files, const char *const *in_paths,
                         const char *const *out_paths, uint64_t *file_counts, swg_stats *stats);
/* Same call with the multi-threaded host parser and writer around swg_filter. */
int swg_filter_paf_host(swg_ctx *ctx, const swg_config *cfg, const char *in_path, const char *out_path,
                        swg_stats *stats);
/* unified_filter::filter_file (src/unified_filter.rs:280-347): sniffs "1 " => .1aln.  The container codec lives in
 * fastga-rs / ONElib, not in sweepga, so a .1aln input is converted through FastGA's own ALNtoPAF when that executable
 * can be found (swg_aln_to_paf below) and the output path ends in ".paf" — the route of the reference's CLI
 * (src/main.rs:737-770); .1aln OUTPUT (write_1aln_filtered, src/unified_filter.rs:158-277) and a .1aln input without the
 * converter => SWG_ERR_UNSUPPORTED.  Parity of this route is unpinned: the reference holds no .1aln vector. */
int swg_filter_file(swg_ctx *ctx, const swg_config *cfg, const char *in_path, const char *out_path,
                    int keep_self, swg_stats *stats);
/* aln_to_paf's fallback (src/main.rs:743-770): runs `ALNtoPAF -x -T<threads> <aln_path>` and writes its standard output
 * (PAF with X-CIGARs) to paf_path.  The executable is $SWG_ALNTOPAF if set, else "ALNtoPAF" on PATH; no shell is involved.
 * SWG_ERR_UNSUPPORTED: no such executable; SWG_ERR_IO: it failed or paf_path cannot be written.  Host only. */
int swg_aln_to_paf(const char *aln_path, const char *paf_path, int threads);

/* ---- multi-GPU sharding helper ------------------------------------------ *
 * Size-balanced (LPT) assignment of genome-pair units (P(q),P(t)) to n_shards.
 * shard_of[i] receives the shard of record i.  Host only, no device needed.     */
int swg_shard_plan(const swg_mappings *host_in, int n_shards, uint32_t *shard_of, uint64_t *shard_sizes);
/* The same rule on unit sizes alone (largest unit first, ties by unit index, onto the least loaded shard, ties by the
 * lowest shard): for drivers that know the unit sizes without holding the table (bench.py generates only its shard). */
int swg_shard_plan_units(uint64_t n_units, const uint64_t *unit_sizes, int n_shards, uint32_t *shard_of_unit,
                         uint64_t *shard_sizes);

/* ---- several GPUs behind one call ----------------------------------------- *
 * One handle owns a context per device.  swg_multi_filter partitions the HOST table by genome-pair unit (swg_shard_plan),
 * filters every shard on its device from its own host thread (swg_filter), and merges the shard results into the caller's
 * arrays with the chain numbers of a single-GPU run (one (A, count) run per unit is all that has to be reconciled, see
 * swg_last_chain_units).  Results do not depend on the number of devices.  NULL + swg_last_error(NULL) when a device
 * cannot be initialised.                                                                                              */
typedef struct swg_multi swg_multi;
swg_multi *swg_multi_create(const int *devices, int n_devices);
void swg_multi_destroy(swg_multi *m);
const char *swg_multi_last_error(const swg_multi *m);
int swg_multi_device_count(const swg_multi *m);
int swg_multi_filter(swg_multi *m, const swg_config *cfg, const swg_mappings *host_in, swg_result *host_out,
                     swg_stats *stats);

const char *swg_version(void);

#ifdef __cplusplus
}
#endif
#endif /* SWEEPGA_B200_H */

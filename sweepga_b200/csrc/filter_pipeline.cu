// filter_pipeline.cu — swg_ctx, the device pipeline that replaces the body of
// PafFilter::apply_filters (reference src/paf_filter.rs:379-747) and its C ABI.
//
// Stage order mirrors the reference (SURVEY.md §8a rows 2..11); run_filter calls one function per stage:
//   K0  prefilter           stage-1 retain                                   paf_filter.rs:384-388
//   GS  primary_sweep       primary plane sweep (closed form when n = inf)   paf_filter.rs:972-1123, plane_sweep_exact.rs
//   K1+sort+K2  order_records  (q,t,strand) grouping + stable sort          paf_filter.rs:761-777
//   K3  chain_groups        best-buddy chaining (huge groups: fixed point)   paf_filter.rs:780-928, union_find.rs
//   K4  chain_table         roots, aggregates, mass/identity filter          paf_filter.rs:449-455
//   O*  order_chains        insertion-order reproduction -> chain_N          SURVEY Appendix B
//   GS                      ... with the scaffold plane sweep                plane_sweep_scaffold.rs:47-251
//   K5  assign_anchors      anchors                                          paf_filter.rs:517-528
//   K6  capture_inversions  inversion capture (inversion_grid: bucketed)     paf_filter.rs:535-597
//   K7  rescue              rescue                                           paf_filter.rs:613-732
#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <thread>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <new>
#include <string>
#include <unordered_map>
#include <vector>

#include "sweepga_b200.h"
#include "common.cuh"
#include "radix_sort.cuh"
#include "scan.cuh"
#include "filter_kernels.cuh"
#include "sweep_tree.cuh"
#include "paf_host.h"

#include <sys/resource.h>
#include <unistd.h>

namespace swg {

struct RangeError { std::string msg; };
struct OomError { size_t bytes; };
struct IoError { std::string msg; };

// ---- generic element-wise launcher (named by Tag so the launch list is readable) ------------
template <class Tag, class F> __global__ void __launch_bounds__(256) k_for(u32 n, F f) {
    u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) f(i);
}
template <class Tag, class F> static inline void launch_for(u32 n, cudaStream_t st, LaunchCounter &lc, F f) {
    if (n == 0) return;
    k_for<Tag, F><<<cdiv(n, 256), 256, 0, st>>>(n, f);
    lc.n++;
}
// the same over a count that lives on the device (no host round trip): fixed grid, grid-stride
template <class Tag, class F> __global__ void __launch_bounds__(256) k_for_dev(const u32 *n_ptr, F f) {
    const u32 n = *n_ptr;
    for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) f(i);
}
template <class Tag, class F> static inline void launch_for_dev(const u32 *n_ptr, int sm_count, cudaStream_t st, LaunchCounter &lc, F f) {
    k_for_dev<Tag, F><<<(u32)sm_count * 8, 256, 0, st>>>(n_ptr, f);
    lc.n++;
}
// add the hits of the active lanes to a counter: one atomic per warp (for rare hits, e.g. the statuses of the inversion capture)
static __device__ __forceinline__ void warp_count_add(u64 *ctr, int slot, bool hit) {
    const u32 am = __activemask();
    const u32 n = __popc(__ballot_sync(am, hit));
    if (n && lane_id() == (u32)(__ffs(am) - 1)) atomicAdd((unsigned long long *)&ctr[slot], (unsigned long long)n);
}
// tags: one per element-wise stage, so that the ncu launch list reads k_for<swg::t_tspace, ...> etc.
struct t_iota; struct t_maxp; struct t_scores; struct t_gkey; struct t_events; struct t_sweep_gather; struct t_sweep_keep;
struct t_gather; struct t_chain_order; struct t_tspace; struct t_segapply; struct t_keys_c2min; struct t_keys_g2min;
struct t_final_k; struct t_invkeys; struct t_invw; struct t_invw2; struct t_invent; struct t_inversion; struct t_anchor_keys; struct t_rescue;

// ---- grow-only HBM arena ----------------------------------------------------------------------
// One block sized for the common path; a call that needs more (general sweeps, degenerate
// inputs) chains extra blocks, and the next reserve() consolidates them into one.
struct Arena {
    struct Block { char *base; size_t cap, off; };
    std::vector<Block> blocks;
    static char *dev_alloc(size_t bytes) {
        char *p = nullptr;
        if (cudaMalloc(&p, bytes) != cudaSuccess) { cudaGetLastError(); throw OomError{bytes}; }
        return p;
    }
    void release() {
        for (auto &b : blocks) cudaFree(b.base);
        blocks.clear();
    }
    void reserve(size_t bytes) {
        size_t total = 0;
        for (auto &b : blocks) total += b.cap;
        if (blocks.size() != 1 || blocks[0].cap < bytes) {
            size_t want = std::max(bytes, total);
            release();
            blocks.push_back(Block{dev_alloc(want), want, 0});
        }
        blocks[0].off = 0;
    }
    template <class T> T *take(size_t n) {
        size_t b = (n * sizeof(T) + 255) & ~(size_t)255;
        if (b == 0) b = 256;
        Block *blk = blocks.empty() ? nullptr : &blocks.back();
        if (!blk || blk->off + b > blk->cap) {
            size_t want = std::max<size_t>(b, (size_t)256 << 20);
            blocks.push_back(Block{dev_alloc(want), want, 0});
            blk = &blocks.back();
        }
        T *p = reinterpret_cast<T *>(blk->base + blk->off);
        blk->off += b;
        return p;
    }
    // stack discipline for temporaries: everything taken after mark() dies at rewind()
    struct Mark { size_t nblocks, off; };
    Mark mark() const { return Mark{blocks.size(), blocks.empty() ? 0 : blocks.back().off}; }
    void rewind(const Mark &m) {
        if (m.nblocks == 0 || blocks.size() < m.nblocks) return;
        for (size_t i = m.nblocks; i < blocks.size(); i++) blocks[i].off = 0; // later blocks stay allocated (grow-only)
        // only the block that was current at mark() can be rewound safely
        if (blocks.size() == m.nblocks) blocks[m.nblocks - 1].off = m.off;
    }
};

} // namespace swg

namespace swg {
// Environment knobs (diagnostics and tests, DESIGN 7b).  Read once per entry point, never cached across calls.
struct Knobs {
    bool force_wide = false, no_fixpoint = false, inv_grid = false, inv_no_diag = false, inv_wide = false, inv_narrow = false, cuda_log = false;
    bool no_fused_keys = false; // SWG_NO_FUSED_KEYS=1: the chain sort keys always come from k_chain_keys
    bool no_group_sort = false; // SWG_NO_GROUP_SORT=1: the record sort always runs the LSD passes (radix_sort.cuh)
    bool sweep_tree_all = false; // SWG_SWEEP_TREE_ALL=1: every group of an n = 1 sweep through the tree (tests)
    bool group_sort_always = false; // SWG_GROUP_SORT_ALWAYS=1: ... never because the rows look ungrouped (tests)
    u32 group_sort_max = 0;     // SWG_GROUP_SORT_MAX: largest group the group sort accepts (default GS_CTA_MAX; tests lower it)
    u32 fixpoint_min = 0;      // 0 = default
    double max_pair_evals = 0; // 0 = no limit (SWG_MAX_PAIR_EVALS)
    int exact_scores = 0;      // SWG_EXACT_SCORES: 0 auto, 1 always, 2 never
    bool stage_timing = false; // SWG_STAGE_TIMING (set, whatever its value): stage events and diagnostic prints
    bool fx_force_collect = false, fixpoint_verify = false; // SWG_FX_FORCE_COLLECT, SWG_FIXPOINT_VERIFY (set, whatever the value)
    int fx_bucket_narrow = 5;        // SWG_FX_BUCKET_NARROW
    int fixpoint_max_rounds = 256;   // SWG_FIXPOINT_MAX_ROUNDS
    u32 tok_long = 4096;             // SWG_TOK_LONG
    bool paf_host_frontend = false;  // SWG_PAF_FRONTEND=host
    u64 paf_batch_bytes = 0;         // SWG_PAF_BATCH_BYTES: cap on the text of one group of swg_filter_paf_batch (0: none)
    u64 paf_batch_memory = 0;        // SWG_PAF_BATCH_MEMORY: device-memory budget of those groups (0: what is free at call start)
};
static Knobs read_knobs() {
    Knobs k;
    auto on = [](const char *n) { const char *v = getenv(n); return v != nullptr && *v && strcmp(v, "0") != 0; };
    k.force_wide = on("SWG_FORCE_WIDE_KEYS");
    k.no_fixpoint = on("SWG_NO_FIXPOINT");
    k.inv_grid = on("SWG_INV_GRID");
    k.inv_no_diag = on("SWG_INV_NO_DIAG");
    k.inv_wide = on("SWG_INV_WIDE");
    k.inv_narrow = on("SWG_INV_NARROW");
    k.no_fused_keys = on("SWG_NO_FUSED_KEYS");
    k.no_group_sort = on("SWG_NO_GROUP_SORT");
    k.group_sort_always = on("SWG_GROUP_SORT_ALWAYS");
    k.sweep_tree_all = on("SWG_SWEEP_TREE_ALL");
    if (const char *v = getenv("SWG_GROUP_SORT_MAX")) k.group_sort_max = (u32)atoi(v);
    if (const char *v = getenv("SWG_LOG_IMPL")) k.cuda_log = strcmp(v, "cuda") == 0;
    if (const char *v = getenv("SWG_FIXPOINT_MIN")) k.fixpoint_min = (u32)atoi(v);
    if (const char *v = getenv("SWG_MAX_PAIR_EVALS")) k.max_pair_evals = atof(v);
    if (const char *v = getenv("SWG_EXACT_SCORES")) k.exact_scores = strcmp(v, "always") == 0 ? 1 : strcmp(v, "never") == 0 ? 2 : 0;
    k.stage_timing = getenv("SWG_STAGE_TIMING") != nullptr;
    k.fx_force_collect = getenv("SWG_FX_FORCE_COLLECT") != nullptr;
    k.fixpoint_verify = getenv("SWG_FIXPOINT_VERIFY") != nullptr;
    if (const char *v = getenv("SWG_FX_BUCKET_NARROW")) k.fx_bucket_narrow = atoi(v);
    if (const char *v = getenv("SWG_FIXPOINT_MAX_ROUNDS")) k.fixpoint_max_rounds = atoi(v);
    if (const char *v = getenv("SWG_TOK_LONG")) k.tok_long = (u32)atoi(v);
    if (const char *v = getenv("SWG_PAF_FRONTEND")) k.paf_host_frontend = strcmp(v, "host") == 0;
    if (const char *v = getenv("SWG_PAF_BATCH_BYTES")) k.paf_batch_bytes = strtoull(v, nullptr, 10);
    if (const char *v = getenv("SWG_PAF_BATCH_MEMORY")) k.paf_batch_memory = strtoull(v, nullptr, 10);
    return k;
}
} // namespace swg

using namespace swg;

struct swg_ctx {
    int device = 0;
    int sm_count = 148;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    cudaStream_t copy_stream = nullptr;          // second stream: the `matches` column is uploaded behind the kernels
    cudaEvent_t ev_copy[2] = {nullptr, nullptr};
    cudaEvent_t ev_sort[2] = {nullptr, nullptr}; // bracket the one-sweep passes of the record sort
    cudaEvent_t ev_pre[2] = {nullptr, nullptr};  // bracket k_prefilter
    cudaEvent_t ev_ctr = nullptr;                // marks an early copy of the counters (read while later kernels still run)
    int sort_passes = 0;
    u64 sort_pairs = 0;
    u64 sort_bytes_per_pair = 24; // of the timed passes: 24 (pairs) or 16 (packed words)
    std::vector<cudaEvent_t> stage_ev;      // SWG_STAGE_TIMING=1: events at stage boundaries of the last call
    std::vector<const char *> stage_name;
    size_t stage_used = 0;
    const u32 *last_keyA = nullptr, *last_keyB = nullptr; // order keys of the kept chains of the last call (in `keys`, not in the scratch arena)
    u64 last_n_chains = 0;
    Arena keys;       // owns last_keyA / last_keyB: they survive later calls that rewind the scratch arena
    const u8 *last_flags = nullptr; // flags[] of the last run_filter (F_ALIVE = passed the stage-1 retain); in the scratch arena
    Arena batch;      // swg_filter_batch: the union of the tables and its results
    bool log_matches_host = false; // swg_create: the device's glibc_log agrees with the host libm's log on the probe set
    bool cudalog_matches_host = false; // ... and CUDA's log() (SWG_LOG_IMPL=cuda) does
    Knobs knobs;      // environment knobs, re-read at the start of every entry point (read_knobs)
    std::vector<double> h_score;   // exact re-rank: host-computed score column
    Arena score_arena;             // ... and its device copy
    Arena arena;      // per-call scratch
    Arena io;         // staging of host SoA for swg_filter
    // swg_prefetch: up to two tables already (being) uploaded, oldest first
    struct Prefetched { bool valid = false; swg_mappings key; swg_mappings dev; swg_result dres; cudaEvent_t ready = nullptr; size_t h2d_bytes = 0; Arena arena; };
    Prefetched pf[2];
    int pf_head = 0, pf_count = 0;
    cudaStream_t up_stream = nullptr;
    bool rows_grouped = false;    // last k_prefilter: the rows come in runs of one (query, target, strand) (aligner order)
    u32 *gtable = nullptr;        // group sort (group_sort.cuh): per possible (query, target, strand) group a counter (u32, cleared
    size_t gtable_entries = 0;    // by every call) and its dense number (u32)
    u64 *h_ctr = nullptr; // pinned mirror of the counters
    std::vector<char *> pin;          // pinned pieces for the file front end (text upload, output download)
    std::vector<cudaEvent_t> pin_ev;
    u32 tok_maxlen = 0;               // longest line of the last tokenised file
    u64 *d_ctr = nullptr;
    std::string err;
    LaunchCounter lc;
};

static std::string g_create_error;

namespace swg {

static void set_err(swg_ctx *c, const std::string &m) { if (c) c->err = m; else g_create_error = m; }

static void stage_mark(swg_ctx *c, const char *name) {
    if (!c->knobs.stage_timing) return;
    if (c->stage_used == c->stage_ev.size()) {
        cudaEvent_t e;
        SWG_CUDA(cudaEventCreate(&e));
        c->stage_ev.push_back(e);
        c->stage_name.push_back(name);
    }
    c->stage_name[c->stage_used] = name;
    SWG_CUDA(cudaEventRecord(c->stage_ev[c->stage_used++], c->stream));
}
static void stage_report(swg_ctx *c) {
    if (c->stage_used < 2) return;
    cudaStreamSynchronize(c->stream);
    fprintf(stderr, "[swg stages]");
    for (size_t i = 0; i + 1 < c->stage_used; i++) {
        float ms = 0;
        cudaEventElapsedTime(&ms, c->stage_ev[i], c->stage_ev[i + 1]);
        fprintf(stderr, " %s %.3f", c->stage_name[i], ms);
    }
    fprintf(stderr, "\n");
}

static void read_counters(swg_ctx *c) {
    SWG_CUDA(cudaMemcpyAsync(c->h_ctr, c->d_ctr, sizeof(u64) * C_COUNT, cudaMemcpyDeviceToHost, c->stream));
    SWG_CUDA(cudaStreamSynchronize(c->stream));
}
// The counters as they are at this point of the stream, without draining it: the copy is marked by an event, the host
// waits for that event only, and kernels enqueued after the copy keep the GPU busy meanwhile.
static void read_counters_begin(swg_ctx *c) {
    SWG_CUDA(cudaMemcpyAsync(c->h_ctr, c->d_ctr, sizeof(u64) * C_COUNT, cudaMemcpyDeviceToHost, c->stream));
    SWG_CUDA(cudaEventRecord(c->ev_ctr, c->stream));
}
static void read_counters_end(swg_ctx *c) { SWG_CUDA(cudaEventSynchronize(c->ev_ctr)); }
static u32 read_u32(swg_ctx *c, const u32 *d) {
    u32 *h = reinterpret_cast<u32 *>(c->h_ctr + C_COUNT);
    SWG_CUDA(cudaMemcpyAsync(h, d, sizeof(u32), cudaMemcpyDeviceToHost, c->stream));
    SWG_CUDA(cudaStreamSynchronize(c->stream));
    return *h;
}

// sort (key,payload) pairs in arena scratch; returns sorted pointers through the references
static void sort_pairs(swg_ctx *c, u64 *&k, u64 *&k2, u32 *&v, u32 *&v2, u32 n, int bits, bool timed = false) {
    if (n == 0) return;
    if (bits > 64) throw RangeError{"sort key wider than 64 bits (too many sequences x coordinate range)"};
    for (int begin = 0; begin < bits; begin += RS_MAX_PASSES * RS_BITS) { // > 8 passes never happens (64 bits)
        RadixSortPlan p = rs_plan(n, begin, bits);
        void *tmp = c->arena.take<char>(p.temp_bytes);
        rs_sort_pairs(p, k, k2, v, v2, tmp, c->stream, c->sm_count, c->lc, timed ? c->ev_sort[0] : nullptr, timed ? c->ev_sort[1] : nullptr);
        if (timed) { c->sort_passes = p.passes; c->sort_pairs = n; }
    }
}
// a key wider than 64 bits as two chained stable sorts, least significant field first: k holds the low field (lo_bits);
// hi(i) = the high field (hi_bits) of item i replaces it for the second sort.  timed: as sort_pairs, for the first sort.
template <class Hi>
static void sort_pairs_wide(swg_ctx *c, u64 *&k, u64 *&k2, u32 *&v, u32 *&v2, u32 n, int lo_bits, int hi_bits, Hi hi, bool timed = false) {
    sort_pairs(c, k, k2, v, v2, n, lo_bits, timed);
    u64 *kk = k;
    const u32 *vv = v;
    launch_for<t_gather>(n, c->stream, c->lc, [=] __device__(u32 p) { kk[p] = hi(vv[p]); });
    sort_pairs(c, k, k2, v, v2, n, hi_bits);
}
// groups of a sorted key: gstart[g] = first position of group g, gid[p] = group of position p, group count to *d_count
static void group_bounds(swg_ctx *c, const u64 *key, int shift, u32 n, u32 *gstart, u32 *gid, u32 *temp, u32 *d_count) {
    scan_flags([=] __device__(u32 p) -> u32 { return (p == 0 || (key[p] >> shift) != (key[p - 1] >> shift)) ? 1u : 0u; },
               [=] __device__(u32 p, u32 ex, u32 v) {
                   if (v) gstart[ex] = p;
                   gid[p] = ex + v - 1;
               },
               n, temp, d_count, c->stream, c->lc);
}

// ---- the group sort (csrc/group_sort.cuh) as one call ---------------------------------------------------------------------
// keys[i] = (group key << shift) | secondary key (< 2^shift); excluded items carry the group key `dead`.  Orders the items by
// (group key, secondary key, index).  On success: out[p] = (group key << ib) | index for the sorted positions p < n_rec,
// gid[p] / gstart[g] / gkey[g] = group of a position, first position and key of a group.  Returns done = false — nothing usable
// written, keys[] untouched — when some group is larger than `limit` (the caller sorts with the LSD passes).
// scratch: n words (sort words); out: n words (may be keys itself); run_of: n u32.  The host reads the counts while the scatter runs;
// with_counters copies the shared counters in the same round trip.
struct GroupSorted {
    bool done = false;
    u32 n_groups = 0, n_rec = 0, n_runs = 0, gmax = 0;
    u32 *gid = nullptr, *gstart = nullptr, *gkey = nullptr;
    const u32 *lists = nullptr; // [3] groups that went through a repair kernel, by size class (device)
    const u32 *d_n_groups = nullptr;
};
static u32 *group_table(swg_ctx *c, u64 entries) { // counters (cleared per use) + dense numbers
    if (c->gtable_entries < entries) {
        if (c->gtable) cudaFree(c->gtable);
        c->gtable = nullptr;
        c->gtable_entries = 0;
        if (cudaMalloc(&c->gtable, entries * 8) != cudaSuccess) { cudaGetLastError(); throw OomError{(size_t)entries * 8}; }
        c->gtable_entries = entries;
    }
    return c->gtable;
}
// largest group the group sort takes (SWG_GROUP_SORT_MAX lowers it)
static u32 group_sort_limit(const Knobs &K) { return K.group_sort_max ? std::min(K.group_sort_max, GS_CTA_MAX) : GS_CTA_MAX; }
static GroupSorted group_sort(swg_ctx *c, const u64 *keys, u64 *scratch, u64 *out, u32 *run_of, u32 n, int shift, GsIndex ix, u32 dead,
                              u64 table_entries, int ib, u32 limit, bool with_counters, u32 *sec_out = nullptr /* n u32: the secondary keys in sorted order */) {
    cudaStream_t st = c->stream;
    Arena &A = c->arena;
    LaunchCounter &lc = c->lc;
    GroupSorted r;
    u32 *gtab = group_table(c, table_entries), *dtab = gtab + table_entries;
    SWG_CUDA(cudaMemsetAsync(gtab, 0, table_entries * 4, st)); // the counters (37 MB for the pairs of 2160 sequences: ~10 us)
    stage_mark(c, "gs_runs");
    // runs of consecutive items with one group key: run index of every item, first item of every run
    u32 *run_start = A.take<u32>((size_t)n + 1), *run_base = A.take<u32>(n);
    u32 *gs_ctr = A.take<u32>(12); // [0] groups, [1] records, [2] largest group; [3] runs; [4..6] list lengths; [7..9] work counters
    SWG_CUDA(cudaMemsetAsync(gs_ctr, 0, 12 * sizeof(u32), st));
    {
        u32 *tmp = A.take<u32>(scan_temp_u32(n));
        scan_flags([=] __device__(u32 i) -> u32 { return (i == 0 || (keys[i] >> shift) != (keys[i - 1] >> shift)) ? 1u : 0u; },
                   [=] __device__(u32 i, u32 ex, u32 v) {
                       if (v) run_start[ex] = i;
                       run_of[i] = ex + v - 1;
                   },
                   n, tmp, gs_ctr + 3, st, lc);
    }
    k_gs_run_base<<<(u32)c->sm_count * 8, 256, 0, st>>>(gs_ctr + 3, run_start, n, keys, shift, ix, dead, gtab, run_base);
    lc.n++;
    stage_mark(c, "gs_scan");
    r.gstart = A.take<u32>((size_t)n + 1);
    r.gkey = A.take<u32>(n);
    r.gid = A.take<u32>(n);
    const u32 tiles = cdiv(table_entries, SC_TILE);
    u64 *gs_status = A.take<u64>((size_t)tiles + 2);
    SWG_CUDA(cudaMemsetAsync(gs_status, 0, sizeof(u64) * ((size_t)tiles + 2), st));
    k_gs_scan<<<tiles, SC_THREADS, 0, st>>>(gtab, dtab, (u32)table_entries, ix, r.gstart, r.gkey, gs_status, reinterpret_cast<u32 *>(gs_status + tiles), gs_ctr);
    lc.n++;
    u32 *h = reinterpret_cast<u32 *>(c->h_ctr + C_COUNT);
    SWG_CUDA(cudaMemcpyAsync(h, gs_ctr, 4 * sizeof(u32), cudaMemcpyDeviceToHost, st));
    if (with_counters) read_counters_begin(c); // the host picks the numbers up while the scatter runs
    else SWG_CUDA(cudaEventRecord(c->ev_ctr, st));
    stage_mark(c, "gs_scatter");
    k_gs_scatter<<<cdiv(n, 256), 256, 0, st>>>(keys, run_of, run_start, run_base, n, shift, ix, dead, ib, gtab, dtab, scratch, r.gid);
    lc.n++;
    read_counters_end(c);
    r.n_groups = h[0]; r.n_rec = h[1]; r.gmax = h[2]; r.n_runs = h[3];
    r.d_n_groups = gs_ctr;
    if (c->knobs.stage_timing) fprintf(stderr, "[swg group sort] records %u runs %u groups %u largest %u\n", r.n_rec, r.n_runs, r.n_groups, r.gmax);
    if (r.n_groups == 0) { r.done = true; return r; }
    if (r.gmax > limit) return r;
    stage_mark(c, "gs_order");
    u32 *list_warp = A.take<u32>(r.n_groups), *list_mid = A.take<u32>(r.n_groups), *list_cta = A.take<u32>(r.n_groups);
    u8 *unsorted = A.take<u8>(r.n_groups);
    u32 *list_ctr = gs_ctr + 4;
    SWG_CUDA(cudaMemsetAsync(unsorted, 0, r.n_groups, st));
    k_gs_emit<<<cdiv(r.n_rec, 256), 256, 0, st>>>(scratch, r.gid, r.gkey, gs_ctr + 1, ib, out, unsorted, sec_out);
    k_gs_groups<<<cdiv(r.n_groups, 256), 256, 0, st>>>(r.n_groups, r.gstart, r.gkey, ib, unsorted, scratch, out, sec_out, list_warp, list_mid, list_cta, list_ctr);
    k_gs_warp<<<(u32)c->sm_count * 8, 256, 0, st>>>(list_warp, list_ctr, gs_ctr + 7, r.gstart, r.gkey, ib, scratch, out, sec_out);
    lc.n += 3;
    if (r.gmax > GS_WARP_MAX) {
        k_gs_mid<<<(u32)c->sm_count * 3, 256, 8 * GS_MID_MAX * sizeof(u64), st>>>(list_mid, list_ctr + 1, gs_ctr + 8, r.gstart, r.gkey, ib, scratch, out, sec_out);
        lc.n++;
    }
    if (r.gmax > GS_MID_MAX) {
        k_gs_cta<<<(u32)c->sm_count * 2, GS_CTA_THREADS, GS_CTA_MAX * sizeof(u64), st>>>(list_cta, list_ctr + 2, gs_ctr + 9, r.gstart, r.gkey, ib, scratch, out, sec_out);
        lc.n++;
    }
    r.lists = list_ctr;
    r.done = true;
    return r;
}

// ---- n = 1 sweep of the piles (csrc/sweep_tree.cuh) -----------------------------------------------------------------------------
struct t_pile_rank; struct t_pile_grp;
static void sweep_piles_n1(swg_ctx *c, const u32 *sitem, const SweepItem *sdata, const u32 *gstart, u32 n_groups, u32 n_sorted,
                           const u32 *big_list, u32 n_big, double thr, u8 *keep) {
    cudaStream_t st = c->stream;
    Arena &A = c->arena;
    LaunchCounter &lc = c->lc;
    stage_mark(c, "pile_events");
    // items of the pile groups
    u32 *boff = A.take<u32>(n_big + 1), *d_tot = A.take<u32>(4);
    u32 *tmp = A.take<u32>(scan_temp_u32(std::max(n_big, 1u)));
    scan_apply([=] __device__(u32 b) -> u32 { const u32 g = big_list[b]; return ((g + 1 < n_groups) ? gstart[g + 1] : n_sorted) - gstart[g]; },
               [=] __device__(u32 b, u32 ex, u32) { boff[b] = ex; }, n_big, tmp, d_tot, st, lc);
    const u32 nb = read_u32(c, d_tot);
    if (nb == 0) return;
    // the event sort below holds 2 * nb pairs, and the radix sort is exact up to 2^30 - 1 pairs (30-bit tile status counts)
    if (nb >= (1u << 29)) throw RangeError{"plane sweep: 2^29 or more mappings in deep piles (the sort of their two events each holds at most 2^30 - 1)"};
    u32 *bitem = A.take<u32>(nb), *bgrp = A.take<u32>(nb);
    k_pile_expand<<<cdiv(nb, 256), 256, 0, st>>>(big_list, boff, n_big, nb, gstart, bitem, bgrp);
    u64 *ek = A.take<u64>(2 * (size_t)nb), *ek2 = A.take<u64>(2 * (size_t)nb), *rk = A.take<u64>(nb), *rk2 = A.take<u64>(nb);
    u32 *ev = A.take<u32>(2 * (size_t)nb), *ev2 = A.take<u32>(2 * (size_t)nb), *rv = A.take<u32>(nb), *rv2 = A.take<u32>(nb);
    k_pile_events<<<cdiv(nb, 256), 256, 0, st>>>(bitem, bgrp, sdata, nb, ek, ev, rk, rv);
    lc.n += 2;
    const int bb = bits_for(n_big);
    sort_pairs(c, ek, ek2, ev, ev2, 2 * nb, 32 + bb);
    // index of every event's position among the distinct (group, position) values
    u32 *upos = A.take<u32>(2 * (size_t)nb);
    {
        u32 *tmp2 = A.take<u32>(scan_temp_u32(2 * nb));
        const u64 *ekc = ek;
        const u32 *evc = ev;
        scan_flags([=] __device__(u32 e) -> u32 { return (ekc[e] != NONE64 && (e == 0 || ekc[e] != ekc[e - 1])) ? 1u : 0u; },
                   [=] __device__(u32 e, u32 ex, u32 v) { upos[evc[e]] = ekc[e] == NONE64 ? NONE32 : ex + v - 1; }, 2 * nb, tmp2, d_tot + 1, st, lc);
    }
    stage_mark(c, "pile_ranks");
    // ranks: stable by score key over items that already are in (group, start, index) order, then stable by group
    sort_pairs(c, rk, rk2, rv, rv2, nb, 64);
    if (n_big > 1) {
        u64 *kk = rk;
        const u32 *vv = rv;
        launch_for<t_pile_grp>(nb, st, lc, [=] __device__(u32 r) { kk[r] = bgrp[vv[r]]; });
        sort_pairs(c, rk, rk2, rv, rv2, nb, bb);
    }
    u32 *rank_of = A.take<u32>(nb);
    {
        const u32 *vv = rv;
        launch_for<t_pile_rank>(nb, st, lc, [=] __device__(u32 r) { rank_of[vv[r]] = r; });
    }
    const u32 *item_of_rank = rv;
    stage_mark(c, "pile_tree");
    u32 size = 1;
    while (size < 2 * nb) size <<= 1;
    u32 *tree = A.take<u32>(2 * (size_t)size), *best = A.take<u32>(2 * (size_t)nb);
    SWG_CUDA(cudaMemsetAsync(tree, 0xFF, sizeof(u32) * 2 * (size_t)size, st));
    k_pile_paint<<<cdiv(nb, 256), 256, 0, st>>>(upos, rank_of, nb, size, tree);
    k_pile_best<<<cdiv(2 * nb, 256), 256, 0, st>>>(tree, 2 * nb, size, best);
    lc.n += 2;
    // runs of one best item
    u32 *run_id = A.take<u32>(2 * (size_t)nb), *run_first = A.take<u32>(2 * (size_t)nb), *run_best = A.take<u32>(2 * (size_t)nb);
    {
        u32 *tmp3 = A.take<u32>(scan_temp_u32(2 * nb));
        scan_flags([=] __device__(u32 i) -> u32 { return (i == 0 || best[i] != best[i - 1]) ? 1u : 0u; },
                   [=] __device__(u32 i, u32 ex, u32 v) {
                       const u32 r = ex + v - 1;
                       run_id[i] = r;
                       if (v) { run_first[r] = i; run_best[r] = best[i]; }
                   },
                   2 * nb, tmp3, d_tot + 2, st, lc);
    }
    stage_mark(c, "pile_verdict");
    k_pile_verdict<<<cdiv(nb, 256), 256, 0, st>>>(bitem, sitem, sdata, upos, rank_of, item_of_rank, run_id, run_first, run_best, d_tot + 2, nb, thr, keep,
                                                   c->d_ctr);
    lc.n++;
    SWG_CUDA(cudaGetLastError());
}

// ---- general plane sweep over arbitrary items (records or chains) ----------------------------
// include == nullptr: all items.  gkey < 2^gb - 1.  keep[] is fully overwritten (0 for excluded).
static void general_sweep_impl(swg_ctx *c, u32 n_items, const u8 *include, u8 include_mask, const u64 *gkey, int gb, int pbits,
                               const u32 *it_start, const u32 *it_end, const double *it_score, u64 n_keep, double thr, u8 *keep) {
    cudaStream_t st = c->stream;
    SWG_CUDA(cudaMemsetAsync(keep, 0, n_items, st));
    if (n_items == 0) return;
    if (gb > 62) throw RangeError{"plane-sweep group key wider than 62 bits"};
    u64 *ek = c->arena.take<u64>(n_items), *ek2 = c->arena.take<u64>(n_items);
    u32 *ev = c->arena.take<u32>(n_items), *ev2 = c->arena.take<u32>(n_items);
    u64 *ctr = c->d_ctr;
    SWG_CUDA(cudaMemsetAsync(ctr + C_TMP0, 0, sizeof(u64), st));
    stage_mark(c, "gs_keys");
    // items in (group, start, item) order; the End events come out of the active set (k_sweep_small).  One sort when
    // the key fits 64 bits, else two chained stable sorts (start first, then the group id).
    const bool wide = (gb + pbits > 64) || c->knobs.force_wide;
    k_sweep_keys<<<std::min<u32>(cdiv(n_items, 256), (u32)c->sm_count * 16), 256, 0, st>>>(n_items, include, include_mask, gkey, wide ? 64 : pbits, it_start, ek, ev, ctr + C_TMP0);
    c->lc.n++;
    int eshift = pbits;
    stage_mark(c, "gs_sort");
    // big grouped inputs (the primary sweeps of a record table in aligner order): the group sort instead of the LSD passes
    const int ib = bits_for(n_items - 1);
    GroupSorted gs;
    if (!wide && !c->knobs.no_group_sort && gb <= 22 && pbits <= 32 && pbits + ib <= 64 && gb + ib <= 64 && n_items >= (1u << 18) &&
        (c->rows_grouped || c->knobs.group_sort_always)) {
        gs = group_sort(c, ek, ek2, ek, ev2, n_items, pbits, GsIndex{0, 0, 0}, 0xFFFFFFFFu, 1ull << gb, ib, group_sort_limit(c->knobs), true);
    }
    if (gs.done) {
        // (sorted item indices: the low bits of ek; t_sweep_gather below writes them to ev)
    } else if (!wide) {
        sort_pairs(c, ek, ek2, ev, ev2, n_items, gb + pbits);
    } else {
        sort_pairs_wide(c, ek, ek2, ev, ev2, n_items, pbits, gb + 1, [=] __device__(u32 i) {
            const bool inc = include ? (include[i] & include_mask) != 0 : true;
            return inc ? gkey[i] : NONE64;
        });
        eshift = 0;
    }
    stage_mark(c, "gs_groups");
    u32 n_inc, n_groups;
    u32 *gstart, *gid;
    SortedIdx sidx{nullptr, ev, 0};
    if (gs.done) {
        n_inc = gs.n_rec;
        if (n_inc != (u32)c->h_ctr[C_TMP0]) throw RangeError{"group sort (sweep): the table counted " + std::to_string(n_inc) + " items"};
        if (n_inc == 0) return;
        n_groups = gs.n_groups;
        gstart = gs.gstart;
        gid = gs.gid;
        sidx = SortedIdx{ek, nullptr, (1ull << ib) - 1};
    } else {
        read_counters(c);
        n_inc = (u32)c->h_ctr[C_TMP0]; // the included items sort first
        if (n_inc == 0) return;
        gstart = c->arena.take<u32>(n_inc + 1);
        gid = c->arena.take<u32>(n_inc);
        u32 *bsum = c->arena.take<u32>(scan_temp_u32(n_inc));
        u32 *d_ng = c->arena.take<u32>(2);
        group_bounds(c, ek, eshift, n_inc, gstart, gid, bsum, d_ng);
        n_groups = read_u32(c, d_ng);
    }
    u32 *ends = n_keep == 1 ? c->arena.take<u32>(n_inc) : nullptr; // interval ends in sorted order (for the running maximum)
    // per-item copies (score key, axis interval) in sorted order: a group becomes one contiguous stream
    SweepItem *sdata = c->arena.take<SweepItem>(n_inc);
    u32 *gflag = c->arena.take<u32>(n_groups);
    SWG_CUDA(cudaMemsetAsync(gflag, 0, sizeof(u32) * (size_t)n_groups, st));
    {
        u32 *evw = gs.done ? ev : nullptr;
        launch_for<t_sweep_gather>(n_inc, st, c->lc, [=] __device__(u32 u) {
            const u32 i = sidx[u];
            if (evw) evw[u] = i;
            if (ends) ends[u] = it_end[i];
            SweepItem d;
            d.skey = score_desc_key(it_score[i]);
            d.start = it_start[i];
            d.end = it_end[i];
            sdata[u] = d;
        });
    }
    u32 *pmax = nullptr;
    if (n_keep == 1) { // running maximum of the interval ends inside every group (bounds the leftward scan of k_sweep_flat1)
        pmax = c->arena.take<u32>(n_inc);
        u32 *tmp = c->arena.take<u32>(scan_temp_u32(n_inc));
        const u32 *gidc = gid;
        scan_segmax([=] __device__(u32 u) -> bool { return u == 0 || gidc[u] != gidc[u - 1]; },
                    [=] __device__(u32 u) -> u32 { return ends[u]; },
                    [=] __device__(u32 u, u32 m) { pmax[u] = m; }, n_inc, tmp, st, c->lc);
    }
    u32 *big_list = c->arena.take<u32>(n_groups + 1);
    u32 *sw_ctr = c->arena.take<u32>(4); // [0] thread-kernel group counter, [1] deep groups, [2] warp-kernel work counter
    SWG_CUDA(cudaMemsetAsync(sw_ctr, 0, 4 * sizeof(u32), st));
    stage_mark(c, "gs_sweep");
    if (n_keep == 1) {
        u32 *rest = c->arena.take<u32>(n_inc);
        const u32 limit = c->knobs.sweep_tree_all ? 0u : SWF_LEFT;
        k_sweep_flat1<<<cdiv(n_inc, 1024), 256, 0, st>>>(ev, sdata, gid, gstart, pmax, n_groups, n_inc, keep, rest, sw_ctr + 3, limit);
        k_sweep_flat1_rest<<<(u32)c->sm_count * 8, 256, 0, st>>>(rest, sw_ctr + 3, ev, sdata, gid, gstart, pmax, n_groups, n_inc, thr, keep, gflag,
                                                                  big_list, sw_ctr + 1, ctr, limit);
        c->lc.n += 2;
        // the groups whose neighbour scans got long (piles) go through the position-parallel tree sweep (sweep_tree.cuh)
        const u32 n_big = read_u32(c, sw_ctr + 1);
        if (n_big) sweep_piles_n1(c, ev, sdata, gstart, n_groups, n_inc, big_list, n_big, thr, keep);
    } else {
        u8 *good = c->arena.take<u8>(n_items), *flagged = c->arena.take<u8>(n_items);
        SWG_CUDA(cudaMemsetAsync(good, 0, n_items, st));
        SWG_CUDA(cudaMemsetAsync(flagged, 0, n_items, st));
        k_sweep_small<<<(u32)c->sm_count * 8, 128, 0, st>>>(ev, sdata, gstart, n_groups, n_inc, n_keep, thr, good, flagged, big_list,
                                                           sw_ctr + 1, sw_ctr, ctr);
        // groups whose pile is deeper than the per-thread array: one warp each, active set in global scratch
        ActEntry *act = c->arena.take<ActEntry>(n_inc + 1);
        k_sweep_groups<<<(u32)c->sm_count * 4, 128, 0, st>>>(ev, sdata, gstart, n_groups, n_inc, n_keep, thr, act, good, flagged, big_list,
                                                            sw_ctr + 1, sw_ctr + 2, ctr);
        c->lc.n += 2;
        const u32 *evc = ev;
        launch_for<t_sweep_keep>(n_inc, st, c->lc, [=] __device__(u32 u) {
            const u32 i = evc[u];
            keep[i] = (good[i] && !flagged[i]) ? 1 : 0;
        });
    }
    stage_mark(c, "gs_done");
    SWG_CUDA(cudaGetLastError());
}

static void general_sweep(swg_ctx *c, u32 n_items, const u8 *include, u8 include_mask, const u64 *gkey, int gb, int pbits,
                          const u32 *it_start, const u32 *it_end, const double *it_score, u64 n_keep, double thr, u8 *keep) {
    Arena::Mark mk = c->arena.mark(); // temporaries are stream-ordered: safe to reuse after the launches are queued
    general_sweep_impl(c, n_items, include, include_mask, gkey, gb, pbits, it_start, it_end, it_score, n_keep, thr, keep);
    c->arena.rewind(mk);
}

} // namespace swg

#include "chain_fixpoint.cuh"

namespace swg {

// score_with_function on the host (plane_sweep_exact.rs:29-86) with the host libm: the exact re-rank's score column
static inline double host_score(int scoring, double identity, u32 qs, u32 qe) {
    const double length = (double)(qe - qs);
    switch (scoring) {
    case 0: return identity <= 0.0 ? -INFINITY : identity;
    case 1: return length <= 0.0 ? -INFINITY : length;
    case 2:
    case 4: return (length <= 0.0 || identity <= 0.0) ? -INFINITY : length * identity;
    default: return (length <= 0.0 || identity <= 0.0) ? -INFINITY : identity * std::log(length);
    }
}

// ================================================================================================
// the pipeline: one function per stage of the list at the top of the file, driven by run_filter
// ================================================================================================
// per-query / per-target limits of the primary sweep (paf_filter.rs:972-1123)
struct Limits { u64 q, t; };
static Limits mapping_limits(const swg_config &cfg) {
    switch (cfg.mapping_filter_mode) {
    case SWG_ONE_TO_ONE: return {1, 1};
    case SWG_ONE_TO_MANY: return {cfg.mapping_max_per_query != SWG_NO_LIMIT ? cfg.mapping_max_per_query : 1, cfg.mapping_max_per_target};
    default: return {cfg.mapping_max_per_query, cfg.mapping_max_per_target};
    }
}

// first-appearance table (hash_insert_min / hash_lookup) for n keys: open addressing over a power of two >= 2n slots (at least
// 1024), every key and value all ones (empty).  Returns the slot mask.
static u32 first_index_table(swg_ctx *c, u64 n, u64 *&hk, u32 *&hv) {
    u32 cap = 1024;
    while ((u64)cap < n * 2) cap <<= 1;
    hk = c->arena.take<u64>(cap);
    hv = c->arena.take<u32>(cap);
    SWG_CUDA(cudaMemsetAsync(hk, 0xFF, sizeof(u64) * cap, c->stream));
    SWG_CUDA(cudaMemsetAsync(hv, 0xFF, sizeof(u32) * cap, c->stream));
    return cap - 1;
}

// the end of every run_filter: stage report, launch count, timings of the record sort and of k_prefilter, the caller's stats
static void finish(swg_ctx *c, swg_stats &S, u64 launches0, swg_stats *stats) {
    stage_mark(c, "end");
    stage_report(c);
    S.gpu_launches = c->lc.n - launches0;
    if (c->sort_passes) { // all work has been synchronised by the last counter read
        float ms = 0;
        cudaStreamSynchronize(c->stream);
        if (cudaEventElapsedTime(&ms, c->ev_sort[0], c->ev_sort[1]) == cudaSuccess) S.ms_sort_passes = ms;
        S.n_sort_passes = (u64)c->sort_passes;
        S.n_sort_pairs = c->sort_pairs;
        S.sort_bytes_per_pair = c->sort_bytes_per_pair;
    }
    if (S.prefilter_bytes_per_record) {
        float ms = 0;
        cudaStreamSynchronize(c->stream);
        if (cudaEventElapsedTime(&ms, c->ev_pre[0], c->ev_pre[1]) == cudaSuccess) S.ms_prefilter = ms;
    }
    if (stats) *stats = S;
}

// ---- K0: stage-1 retain (k_prefilter) ----------------------------------------------------------
struct Prefiltered {
    u8 *flags;
    u64 *hk; u32 *hv; u32 hmask;                 // genome pair -> first record index
    uint4 *rec4 = nullptr;                       // packed coordinates (scaffolding only, like the sort buffers)
    u64 *keys = nullptr, *keys2 = nullptr;
    u32 *vals = nullptr, *vals2 = nullptr;
    bool fused_keys;           // k_prefilter wrote the chain sort keys into keys / vals
    bool gsort;                // the record sort may take the group sort: its table of g_entries groups fits
    u64 g_entries;
    u64 n_alive, zlq, zlt;     // records alive; ... with an empty query / target interval
    u32 maxcoord;
    int sb, cb, pb;            // bits of a sequence id, a coordinate, a genome-prefix id
};
static Prefiltered prefilter(swg_ctx *c, const swg_config &cfg, const DevIn &in, const Limits &lim, u8 *status, u32 *chain_id,
                             cudaEvent_t ev_matches, swg_stats &S) {
    cudaStream_t st = c->stream;
    const Knobs &K = c->knobs;
    LaunchCounter &lc = c->lc;
    const u32 N = in.n;
    c->arena.reserve((size_t)N * 400 + (64u << 20));
    Arena &A = c->arena;
    u64 *ctr = c->d_ctr;
    SWG_CUDA(cudaMemsetAsync(ctr, 0, sizeof(u64) * C_COUNT, st));

    stage_mark(c, "prefilter");
    Prefiltered P;
    P.flags = A.take<u8>(N);
    c->last_flags = P.flags;
    // distinct genome pairs <= min(N, nP^2); table of 2x that, power of two
    u32 *d_maxp = A.take<u32>(2);
    SWG_CUDA(cudaMemsetAsync(d_maxp, 0, 2 * sizeof(u32), st));
    launch_for<t_maxp>(in.n_seq, st, lc, [=] __device__(u32 s) { atomicMax(&d_maxp[0], in.P[s]); atomicMax(&d_maxp[1], in.P2[s]); });
    u32 maxP, maxP2;
    {   // both in one round trip; the result arrays are cleared while the host waits for it
        u32 *h = reinterpret_cast<u32 *>(c->h_ctr + C_COUNT);
        SWG_CUDA(cudaMemcpyAsync(h, d_maxp, 2 * sizeof(u32), cudaMemcpyDeviceToHost, st));
        SWG_CUDA(cudaEventRecord(c->ev_ctr, st));
        SWG_CUDA(cudaMemsetAsync(status, 0, N, st));
        SWG_CUDA(cudaMemsetAsync(chain_id, 0, sizeof(u32) * (size_t)N, st));
        SWG_CUDA(cudaEventSynchronize(c->ev_ctr));
        maxP = h[0];
        maxP2 = h[1];
    }
    if (maxP >= in.n_seq || maxP2 >= in.n_seq) throw RangeError{"genome prefix id >= n_seq (prefix ids must be dense)"};
    P.hmask = first_index_table(c, std::min<u64>((u64)N, (u64)(maxP + 1) * (maxP + 1)), P.hk, P.hv);
    if (cfg.scaffold_gap != 0) P.rec4 = A.take<uint4>(N);
    // swg_filter sends `matches` — and `block_length`, when the retain does not test it — behind the other columns: k_prefilter waits
    // for them only if it derives the identity from them
    if (ev_matches && !in.identity && !(cfg.min_identity <= 0.0)) SWG_CUDA(cudaStreamWaitEvent(st, ev_matches, 0));
    // The chain sort keys can be written by the same pass when the primary sweep is the closed form (no per-axis limit): then
    // kept == alive unless an alive record has an empty interval (checked below; k_chain_keys redoes the keys in that case).
    P.sb = bits_for(in.n_seq); // ids < n_seq <= 2^sb - 1: the all-ones pattern stays free for dead keys
    P.fused_keys = cfg.scaffold_gap != 0 && lim.q == SWG_KEEP_ALL && lim.t == SWG_KEEP_ALL && !K.force_wide && 2 * P.sb + 1 <= 32 &&
                   !K.no_fused_keys;
    if (cfg.scaffold_gap != 0) { P.keys = A.take<u64>(N); P.keys2 = A.take<u64>(N); P.vals = A.take<u32>(N); P.vals2 = A.take<u32>(N); }
    // The record sort as a counting sort by group (group_sort.cuh) when the table of all possible groups fits.
    P.g_entries = 2ull * in.n_seq * in.n_seq;
    P.gsort = cfg.scaffold_gap != 0 && !K.force_wide && !K.no_group_sort && P.g_entries <= GS_MAX_TABLE && 2 * P.sb + 1 <= 31;
    if (P.gsort) {
        try { group_table(c, P.g_entries); } // (up to 512 MB for ~5800 sequences) no room: the LSD passes need no table
        catch (const OomError &) { P.gsort = false; }
    }
    SWG_CUDA(cudaEventRecord(c->ev_pre[0], st));
    if (P.fused_keys)
        k_prefilter<true><<<cdiv(N, 256), 256, 0, st>>>(in, cfg.min_block_length, cfg.min_identity, cfg.keep_self, P.flags, ctr, P.hk, P.hv,
                                                        P.hmask, P.rec4, P.sb, P.keys, P.vals);
    else k_prefilter<false><<<cdiv(N, 256), 256, 0, st>>>(in, cfg.min_block_length, cfg.min_identity, cfg.keep_self, P.flags, ctr, P.hk, P.hv,
                                                          P.hmask, P.rec4);
    SWG_CUDA(cudaEventRecord(c->ev_pre[1], st));
    {   // algorithmic bytes of the launch per record: ids 8, coordinates 16, block length 4, strand 1 (+ matches 4 / identity 8 when
        // the identity test needs them) read; flags 1 (+ packed coordinates 16, + key 8 and index 4 when the pass writes the keys) written
        const bool need_id = in.identity != nullptr || !(cfg.min_identity <= 0.0);
        S.prefilter_bytes_per_record = 29 + (need_id ? (in.identity ? 8 : 4) : 0) + 1 + (P.rec4 ? 16 : 0) + (P.fused_keys ? 12 : 0);
    }
    lc.n++;
    read_counters(c);
    if (c->h_ctr[C_BAD])
        throw RangeError{"a record that passes the length / self / identity retain has end < start, a coordinate beyond the u32 table, or a sequence id >= n_seq"};
    P.n_alive = c->h_ctr[C_ALIVE], P.zlq = c->h_ctr[C_ZLQ], P.zlt = c->h_ctr[C_ZLT];
    c->rows_grouped = (c->h_ctr[C_RUNS] - std::min<u64>(c->h_ctr[C_RUNS], N / 32)) * 2 <= (u64)N;
    P.maxcoord = (u32)c->h_ctr[C_MAXCOORD];
    S.n_stage1 = P.n_alive;
    P.cb = bits_for(P.maxcoord);
    P.pb = bits_for(maxP); // genome-prefix ids of the partner: usually far fewer bits than a sequence id, and one sort pass less
    return P;
}

// ---- GS: primary plane sweep (paf_filter.rs:972-1123) ------------------------------------------
struct Kept { u8 *q = nullptr, *t = nullptr; }; // per record: kept by the query / target axis sweep; nullptr: that sweep keeps all
static Kept primary_sweep(swg_ctx *c, const swg_config &cfg, const DevIn &in, const Prefiltered &P, const Limits &lim,
                          cudaEvent_t ev_matches) {
    cudaStream_t st = c->stream; LaunchCounter &lc = c->lc; Arena &A = c->arena;
    const bool cuda_log = c->knobs.cuda_log;
    const u32 N = in.n;
    const int pb = P.pb;
    stage_mark(c, "primary_sweep");
    Kept kept;
    const bool need_q = P.n_alive > 1 && (lim.q != SWG_KEEP_ALL || P.zlq > 0);
    const bool need_t = P.n_alive > 1 && (lim.t != SWG_KEEP_ALL || P.zlt > 0);
    if (!need_q && !need_t) return kept;
    double *rscore = A.take<double>(N);
    const int scoring = cfg.scoring_function;
    if (ev_matches && !in.identity && !in.score) SWG_CUDA(cudaStreamWaitEvent(st, ev_matches, 0));
    launch_for<t_scores>(N, st, lc, [=] __device__(u32 i) {
        rscore[i] = in.score ? in.score[i] : score_fn(scoring, rec_identity(in, i), in.qs[i], in.qe[i], cuda_log);
    });
    u64 *gk = A.take<u64>(N);
    for (int axis = 0; axis < 2; axis++) {
        if (axis == 0 ? !need_q : !need_t) continue;
        launch_for<t_gkey>(N, st, lc, [=] __device__(u32 i) {
            u32 a = axis == 0 ? in.qid[i] : in.tid[i], b = axis == 0 ? in.tid[i] : in.qid[i];
            gk[i] = ((u64)a << pb) | in.P[b];
        });
        u8 *keep = A.take<u8>(N);
        general_sweep(c, N, P.flags, F_ALIVE, gk, P.sb + pb, P.cb, axis == 0 ? in.qs : in.ts, axis == 0 ? in.qe : in.te, rscore,
                      axis == 0 ? lim.q : lim.t, cfg.overlap_threshold, keep);
        (axis == 0 ? kept.q : kept.t) = keep;
    }
    return kept;
}

// ---- K1 + sort + K2: group by (q,t,strand), stable order by query_start; the packed coordinates in that order -------------
struct Ordered {
    u32 n_m = 0;                         // records kept by the primary sweep = sorted positions
    const u64 *skey = nullptr;           // group key of a sorted position = skey >> gshift
    int gshift = 0;
    SortedIdx sidx{nullptr, nullptr, 0}; // record index of a sorted position
    u32 n_groups = 0;
    const u32 *gstart = nullptr, *gid = nullptr;
    const uint4 *srec = nullptr;         // packed coordinates of the sorted positions
    const u32 *gs_lists = nullptr;       // group sort: [3] groups that had to be ordered, by size class (diagnostic)
    u32 fx_min = 0;                      // groups of at least fx_min positions are chained by the fixed-point iteration
};
static Ordered order_records(swg_ctx *c, const swg_config &cfg, const DevIn &in, const Prefiltered &P, const Kept &kept, swg_stats &S) {
    cudaStream_t st = c->stream; LaunchCounter &lc = c->lc; Arena &A = c->arena;
    const Knobs &K = c->knobs;
    const u32 N = in.n;
    u64 *ctr = c->d_ctr;
    u8 *flags = P.flags;
    const uint4 *rec4 = P.rec4;
    const u8 *keep_q = kept.q, *keep_t = kept.t;
    u64 *keys = P.keys, *keys2 = P.keys2;
    u32 *vals = P.vals, *vals2 = P.vals2;
    const int sb = P.sb, cb = P.cb;
    stage_mark(c, "keys+sort");
    int gshift = cb; // group id of a sorted position = skey >> gshift
    const int kb = 2 * sb + 1 + cb;
    // The packed LSD sort keeps the key from bit c0 upwards; the group key starts at bit cb, so c0 > cb (many sequences, narrow
    // coordinates, 2^24 or more records) would cut group bits: such inputs take the two-stage path as well.
    const bool wide = kb > 64 || K.force_wide || rs_packed_c0(kb, bits_for(N - 1)) > cb;
    SortedIdx sidx{nullptr, nullptr, 0};
    const u64 *skey = nullptr;
    bool kept_is_alive = false;   // the keys came from k_prefilter: kept == alive, nobody counted C_KEPT_M
    bool groups_done = false;     // gid / gstart / group count already produced (group sort)
    u32 gs_gmax = 0;              // group sort: its largest group
    const u32 *gs_lists = nullptr; // ... the groups it had to order, by size class
    u32 n_groups = 0;
    u32 *gstart = nullptr, *gid = nullptr;
    u32 *d_ng = A.take<u32>(1);   // group count (k_chain_work_estimate)
    if (!wide) {
        const int ib = bits_for(N - 1);
        // the keys written by k_prefilter<true> stand if no sweep ran (kept == alive)
        const bool fused_ok = P.fused_keys && !keep_q && !keep_t && P.zlq == 0 && P.zlt == 0;
        // ... for the LSD passes additionally every digit consumed up to the packing pass must lie inside the coordinate field
        // (the gap of the layout is closed by the packing pass)
        const bool fused_lsd_ok = fused_ok && rs_packed_c0(kb, ib) > 0 && rs_packed_c0(kb, ib) <= cb;
        bool lsd = true, fused_keys = fused_lsd_ok;
        int key_shift = cb; // keys[] = (group key << key_shift) | query_start
        // rows in no particular order (runs of ~1 record: every step of the group sort turns into random accesses, ~1.6x the
        // LSD passes on a shuffled 20 M table) go through the LSD passes
        const bool grouped_rows = c->rows_grouped || K.group_sort_always;
        if (P.gsort && grouped_rows) {
            if (fused_ok) { key_shift = 32; kept_is_alive = true; }
            else {
                k_chain_keys<<<cdiv(N, 256), 256, 0, st>>>(in, flags, keep_q, keep_t, sb, cb, keys, vals, ctr);
                lc.n++;
            }
            const GroupSorted gs = group_sort(c, keys, keys2, keys /* the keys have done their duty by then */, vals2, N, key_shift,
                                              GsIndex{1, sb, in.n_seq}, (1u << (2 * sb + 1)) - 1, P.g_entries, ib, group_sort_limit(K), true);
            if (gs.n_rec != (kept_is_alive ? (u32)P.n_alive : (u32)c->h_ctr[C_KEPT_M])) throw RangeError{"group sort: the table counted " + std::to_string(gs.n_rec) + " records"};
            if (gs.done) {
                lsd = false;
                if (gs.n_groups) {
                    SWG_CUDA(cudaMemcpyAsync(d_ng, gs.d_n_groups, sizeof(u32), cudaMemcpyDeviceToDevice, st));
                    n_groups = gs.n_groups;
                    gstart = gs.gstart;
                    gid = gs.gid;
                    skey = keys;
                    sidx.w = keys;
                    sidx.mask = (1ull << ib) - 1;
                    gshift = ib;
                    groups_done = true;
                    gs_lists = gs.lists;
                    gs_gmax = gs.gmax;
                }
            } else {
                // some group is larger than one CTA sorts: the LSD passes take over (the keys are still in place)
                if (key_shift == 32 && !fused_lsd_ok) { // the gap layout does not suit the LSD passes of this key width
                    k_chain_keys<<<cdiv(N, 256), 256, 0, st>>>(in, flags, keep_q, keep_t, sb, cb, keys, vals, ctr);
                    lc.n++;
                    kept_is_alive = false;
                    fused_keys = false;
                    read_counters(c);
                } else fused_keys = key_shift == 32;
            }
        } else {
            kept_is_alive = fused_keys;
            if (!fused_keys) {
                k_chain_keys<<<cdiv(N, 256), 256, 0, st>>>(in, flags, keep_q, keep_t, sb, cb, keys, vals, ctr);
                lc.n++;
            }
        }
        if (lsd) {
            read_counters_begin(c); // the survivor count is final here; the host picks it up while the sort runs
            // the packed sort (radix_sort.cuh): once the key bits still to be sorted and the index fit one word, the passes
            // move 8 B per record instead of 12 B; the result holds the index and the key from bit c0 upwards
            RadixSortPlan p = rs_plan(N, 0, kb);
            void *tmp = A.take<char>(p.temp_bytes);
            const PackedSort ps = rs_sort_packed(N, kb, ib, keys, keys2, vals, vals2, tmp, p, st, c->sm_count, lc, c->ev_sort[0], c->ev_sort[1],
                                                 fused_keys ? cb : 0);
            c->sort_passes = ps.timed_passes; // the events bracket the packed-word passes
            c->sort_pairs = N;
            c->sort_bytes_per_pair = ps.timed_bytes_per_pair;
            skey = ps.packed;
            sidx.w = ps.packed;
            sidx.mask = (1ull << ib) - 1;
            gshift = ib + cb - ps.c0;
            read_counters_end(c);
        }
    } else {
        // key wider than 64 bits (hundreds of thousands of sequences): sorted by query_start, then by the (query,target,strand)
        // group id; skey then holds the group id alone
        u64 *gk = A.take<u64>(N);
        {
            u64 *kk = keys;
            u32 *vv = vals;
            launch_for<t_gkey>(N, st, lc, [=] __device__(u32 i) {
                const bool kept = (flags[i] & F_ALIVE) && (!keep_q || keep_q[i]) && (!keep_t || keep_t[i]);
                const u64 sbit = in.strand[i] == '+' ? 0 : 1;
                gk[i] = kept ? ((((u64)in.qid[i] << sb) | in.tid[i]) << 1 | sbit) : NONE64;
                kk[i] = in.qs[i];
                vv[i] = i;
                u32 am = __activemask();
                u32 cnt = __popc(__ballot_sync(am, kept));
                if (cnt && (threadIdx.x & 31) == (u32)(__ffs(am) - 1)) atomicAdd((unsigned long long *)&ctr[C_KEPT_M], (unsigned long long)cnt);
            });
        }
        sort_pairs_wide(c, keys, keys2, vals, vals2, N, cb, 2 * sb + 2, [=] __device__(u32 i) { return gk[i]; }, true);
        gshift = 0;
        skey = keys;
        sidx.v = vals;
        read_counters(c);
    }
    const u32 n_m = kept_is_alive ? (u32)P.n_alive : (u32)c->h_ctr[C_KEPT_M]; // keys of k_prefilter: kept == alive (nobody counted)
    S.n_after_sweep = n_m;
    S.score_near_ties = c->h_ctr[C_NEAR_TIES];
    if (n_m == 0) return Ordered{};
    stage_mark(c, "groups+gather");
    uint4 *srec = A.take<uint4>(n_m);
    if (!groups_done) {
        gstart = A.take<u32>(n_m + 1);
        gid = A.take<u32>(n_m);
        group_bounds(c, skey, gshift, n_m, gstart, gid, A.take<u32>(scan_temp_u32(n_m)), d_ng);
    }
    // groups of at least fx_min positions are chained by the fixed-point iteration (SWG_NO_FIXPOINT=1: by the warp walk)
    const u32 fx_min = K.no_fixpoint ? NONE32 : (K.fixpoint_min ? K.fixpoint_min : FX_MIN_GROUP);
    if (groups_done && gs_gmax < fx_min && !(K.max_pair_evals > 0)) {
        // the group sort has told the host the group count and the largest group: no huge group, nothing to estimate, no round trip
        launch_for<t_gather>(n_m, st, lc, [=] __device__(u32 p) { srec[p] = __ldg(&rec4[sidx[p]]); });
    } else {
        // group count, positions in huge groups and a rough count of the candidate evaluations ahead (SWG_MAX_PAIR_EVALS, if
        // set, refuses an input beyond it; by default nothing is refused: the reference runs such piles to completion too).
        // The host picks the numbers up while the gather below runs.
        if (K.max_pair_evals > 0) k_chain_work_estimate<true><<<(u32)c->sm_count * 8, 256, 0, st>>>(rec4, sidx, gstart, d_ng, n_m, cfg.scaffold_gap, fx_min, ctr);
        else k_chain_work_estimate<false><<<(u32)c->sm_count * 8, 256, 0, st>>>(rec4, sidx, gstart, d_ng, n_m, cfg.scaffold_gap, fx_min, ctr);
        lc.n++;
        u32 *h = reinterpret_cast<u32 *>(c->h_ctr + C_COUNT);
        SWG_CUDA(cudaMemcpyAsync(h, d_ng, sizeof(u32), cudaMemcpyDeviceToHost, st)); // group count and estimate in one round trip
        read_counters_begin(c);
        // post-sort gather of the packed coordinates (flat, one thread per position: all gathers of a warp in flight at once;
        // fused into the scan above it ran 5x slower: a scan thread owns eight CONSECUTIVE positions, so neither side coalesces).
        // block_length / matches are not copied: the aggregate pass gathers them itself.
        launch_for<t_gather>(n_m, st, lc, [=] __device__(u32 p) { srec[p] = __ldg(&rec4[sidx[p]]); });
        read_counters_end(c);
        n_groups = *h;
        if (K.max_pair_evals > 0 && (double)c->h_ctr[C_WORK] > K.max_pair_evals)
            throw RangeError{"chaining would need ~" + std::to_string((double)c->h_ctr[C_WORK]) +
                             " candidate evaluations (dense pile), more than SWG_MAX_PAIR_EVALS"};
    }
    return Ordered{n_m, skey, gshift, sidx, n_groups, gstart, gid, srec, gs_lists, fx_min};
}

// ---- K3: best-buddy chaining (claims -> sequential resolve of the dirty groups; huge groups: the fixed point) -------------
struct Chained {
    const u32 *pred;        // best predecessor of every sorted position
    const u32 *root_preset; // roots of the positions of huge groups (fixed-point chaining), NONE32 elsewhere; nullptr: none
    u32 n_huge;             // positions in huge groups (also selects the bucketed inversion capture)
    const u32 *bb_ctr;      // [0] ordinary dirty groups, [2] large/dense dirty groups (diagnostic)
};
static Chained chain_groups(swg_ctx *c, const swg_config &cfg, const Ordered &O, u32 maxcoord) {
    cudaStream_t st = c->stream; LaunchCounter &lc = c->lc; Arena &A = c->arena;
    const u32 n_m = O.n_m, n_groups = O.n_groups, fx_min = O.fx_min;
    const u32 *gstart = O.gstart, *gid = O.gid;
    const uint4 *srec = O.srec;
    const u64 *skey = O.skey;
    const int gshift = O.gshift;
    stage_mark(c, "chaining");
    u64 *bps = A.take<u64>(n_m);     // best_pred_score: only the dirty groups touch it
    u32 *pred = A.take<u32>(n_m);    // best_pred_idx
    u32 *grp_dirty = A.take<u32>(n_groups);
    u32 *work = A.take<u32>(n_groups), *work_big = A.take<u32>(n_groups);
    u32 *bb_ctr = A.take<u32>(4); // [0] #ordinary dirty groups, [1] their work counter, [2] #large/dense dirty groups, [3] their work counter
    u32 *root_preset = nullptr;
    SWG_CUDA(cudaMemsetAsync(bb_ctr, 0, 4 * sizeof(u32), st));
    SWG_CUDA(cudaMemsetAsync(grp_dirty, 0, sizeof(u32) * (size_t)n_groups, st));
    SWG_CUDA(cudaMemsetAsync(pred, 0xFF, sizeof(u32) * (size_t)n_m, st));
    // claims; a group with a conflict puts itself on a work list: ordinary (thread per group) or large/dense (warp per group:
    // more than RES_THREAD_MAX positions or an expected window > 64 candidates)
    k_chain_candidates<false><<<cdiv(n_m, 256), 256, 0, st>>>(srec, skey, gid, gstart, n_groups, n_m, gshift, cfg.scaffold_gap, nullptr, pred, grp_dirty,
                                                               nullptr, nullptr, c->h_ctr[C_HUGE] ? fx_min : NONE32, work, work_big, bb_ctr);
    lc.n++;
    stage_mark(c, "ch_worklists");
    auto is_huge = [=] __device__(u32 g) -> bool {
        const u32 s0 = gstart[g], e0 = (g + 1 < n_groups) ? gstart[g + 1] : n_m;
        return e0 - s0 >= fx_min;
    };
    // the redone groups need their candidate records: a second candidate pass over the listed groups only (ordinary data: a
    // few hundred groups; writing all 16 B records in the first pass cost more than it saved)
    Cand *cand = A.take<Cand>(n_m); // unconstrained arg-min of every position of the groups that are redone (dirty / huge)
    k_chain_candidates_groups<<<(u32)c->sm_count * 4, 256, 0, st>>>(srec, skey, gstart, n_groups, n_m, gshift, cfg.scaffold_gap, cand, work, bb_ctr,
                                                                   work_big, bb_ctr + 2);
    lc.n++;
    stage_mark(c, "ch_resolve");
    // enough threads to hide the dependent-load latency of a step, few enough that every group's lines stay in L1/L2
    k_chain_resolve<<<(u32)c->sm_count * 4, 128, 0, st>>>(cand, srec, skey, gstart, n_groups, n_m, work, bb_ctr, gshift, cfg.scaffold_gap,
                                                          bps, pred, bb_ctr + 1);
    k_chain_resolve_warp<<<(u32)c->sm_count * 4, 128, 0, st>>>(cand, srec, skey, gstart, n_groups, n_m, work_big, bb_ctr + 2, gshift,
                                                              cfg.scaffold_gap, bps, pred, bb_ctr + 3);
    lc.n += 2;
    const u32 n_huge = (u32)c->h_ctr[C_HUGE];
    if (n_huge) {
        stage_mark(c, "ch_fixpoint");
        u32 *hpos = A.take<u32>(n_huge);
        u32 *d_nh = A.take<u32>(1);
        u32 *bsum = A.take<u32>(scan_temp_u32(n_m));
        root_preset = A.take<u32>(n_m);
        SWG_CUDA(cudaMemsetAsync(root_preset, 0xFF, sizeof(u32) * (size_t)n_m, st));
        scan_flags([=] __device__(u32 p) -> u32 { return is_huge(gid[p]) ? 1u : 0u; },
                   [=] __device__(u32 p, u32 ex, u32 v) { if (v) hpos[ex] = p; }, n_m, bsum, d_nh, st, lc);
        if (!chain_fixpoint(c, n_huge, hpos, srec, skey, gshift, gid, gstart, n_groups, n_m, cfg.scaffold_gap, root_preset, bsum, maxcoord)) {
            // a dependency chain longer than the round limit: the huge groups go through the sequential warp walk after all
            // (it resets the groups' pred / best_pred_score itself; root_preset is untouched).  The walk starts from the
            // candidate records of their positions (position-parallel).
            k_chain_candidates<true><<<(u32)c->sm_count * 16, 256, 0, st>>>(srec, skey, gid, gstart, n_groups, n_m, gshift, cfg.scaffold_gap, cand, nullptr,
                                                                             nullptr, hpos, d_nh);
            lc.n++;
            SWG_CUDA(cudaMemsetAsync(bb_ctr + 2, 0, 2 * sizeof(u32), st));
            scan_flags([=] __device__(u32 g) -> u32 { return is_huge(g) ? 1u : 0u; },
                       [=] __device__(u32 g, u32 ex, u32 v) { if (v) work_big[ex] = g; }, n_groups, bsum, bb_ctr + 2, st, lc);
            k_chain_resolve_warp<<<(u32)c->sm_count * 4, 128, 0, st>>>(cand, srec, skey, gstart, n_groups, n_m, work_big, bb_ctr + 2, gshift,
                                                                      cfg.scaffold_gap, bps, pred, bb_ctr + 3);
            lc.n++;
        }
    }
    return Chained{pred, root_preset, n_huge, bb_ctr};
}

// ---- K4: roots + dense chain numbers (k_chain_number), aggregates, the mass/identity filter, the passing chains sorted -----
struct Chains {
    const u32 *chain_of; // chain number of every sorted position
    ChainTable ct;       // C rows
    u32 C, C1;           // chains; chains that pass the mass/identity filter
    const u64 *okey;     // the C1 passing chains in order: their order keys (first index of the genome pair, of the group) ...
    const u32 *oval;     // ... and chain numbers
    u64 pass_zero;       // passing chains with an empty query or target interval
};
static Chains chain_table(swg_ctx *c, const swg_config &cfg, const DevIn &in, const Prefiltered &P, const Ordered &O, const Chained &chained,
                          cudaEvent_t ev_matches, bool exact_host, swg_stats &S) {
    cudaStream_t st = c->stream; LaunchCounter &lc = c->lc; Arena &A = c->arena;
    const bool cuda_log = c->knobs.cuda_log;
    u64 *ctr = c->d_ctr;
    const u32 n_m = O.n_m;
    const u64 *skey = O.skey;
    const int gshift = O.gshift;
    const u32 *gid = O.gid;
    const int sb = P.sb;
    stage_mark(c, "ch_number");
    // The table is sized for the worst case (every position its own chain) and each row is cleared by the kernel that numbers
    // its chain, so the aggregate pass can start before the host knows the chain count (it reads it while that pass runs).
    u32 *chain_of = A.take<u32>(n_m);  // chain number of every sorted position (cross-tile marks resolved by the aggregate pass)
    u32 *head_pos = A.take<u32>(n_m);  // compacted head positions (C of them)
    u32 *grp_minidx = A.take<u32>(O.n_groups); // per GROUP: min original index over its members (first appearance of the group)
    u32 *d_cnt = A.take<u32>(2);       // [0] chains, [1] passing chains
    SWG_CUDA(cudaMemsetAsync(grp_minidx, 0xFF, sizeof(u32) * (size_t)O.n_groups, st));
    ChainTable ct;
    ct.pos = head_pos; ct.qid = A.take<u32>(n_m); ct.tid = A.take<u32>(n_m); ct.fwd = A.take<u8>(n_m);
    ct.qs = A.take<u32>(n_m); ct.qe = A.take<u32>(n_m); ct.ts = A.take<u32>(n_m); ct.te = A.take<u32>(n_m);
    ct.wid = A.take<double>(n_m); ct.pass = A.take<u8>(n_m); ct.k = A.take<u32>(n_m);
    ChainDense cd;
    cd.qmin = ct.qs; cd.qmax = ct.qe; cd.tmin = ct.ts; cd.tmax = ct.te; cd.k = ct.k;
    cd.sum_matches = A.take<u64>(n_m); cd.sum_block = A.take<u64>(n_m);
    {
        const u32 tiles = cdiv(n_m, CR_TILE);
        u64 *cn_status = A.take<u64>(tiles + 1);
        u32 *cn_ctr = A.take<u32>(2);
        SWG_CUDA(cudaMemsetAsync(cn_status, 0, sizeof(u64) * (size_t)(tiles + 1), st));
        SWG_CUDA(cudaMemsetAsync(cn_ctr, 0, 2 * sizeof(u32), st));
        if (chained.root_preset) k_chain_number<true><<<tiles, CR_THREADS, 0, st>>>(chained.pred, chained.root_preset, n_m, chain_of, head_pos, cn_status, cn_ctr, d_cnt, cd);
        else k_chain_number<false><<<tiles, CR_THREADS, 0, st>>>(chained.pred, nullptr, n_m, chain_of, head_pos, cn_status, cn_ctr, d_cnt, cd);
        lc.n++;
    }
    {   // the chain count (and, as diagnostics, how many groups had to be redone sequentially) travels while the aggregate runs
        u32 *h = reinterpret_cast<u32 *>(c->h_ctr + C_COUNT);
        SWG_CUDA(cudaMemcpyAsync(h, d_cnt, sizeof(u32), cudaMemcpyDeviceToHost, st));
        SWG_CUDA(cudaMemcpyAsync(h + 2, chained.bb_ctr, 4 * sizeof(u32), cudaMemcpyDeviceToHost, st));
        if (O.gs_lists) SWG_CUDA(cudaMemcpyAsync(h + 6, O.gs_lists, 3 * sizeof(u32), cudaMemcpyDeviceToHost, st));
        SWG_CUDA(cudaEventRecord(c->ev_ctr, st));
    }
    if (ev_matches) SWG_CUDA(cudaStreamWaitEvent(st, ev_matches, 0)); // first use of in.matches
    k_chain_aggregate<<<cdiv(n_m, 256), 256, 0, st>>>(O.srec, in.blen, in.matches, O.sidx, gid, chain_of, n_m, cd, grp_minidx);
    lc.n++;
    SWG_CUDA(cudaEventSynchronize(c->ev_ctr));
    u32 C;
    {
        const u32 *h = reinterpret_cast<const u32 *>(c->h_ctr + C_COUNT);
        C = h[0];
        S.n_dirty_groups = (u64)h[2] + h[4];
        if (O.gs_lists) S.n_unsorted_groups = (u64)h[6] + h[7] + h[8];
    }
    stage_mark(c, "chain_table");
    S.n_chains = C;
    // exact re-rank: ln(gap) of every chain from the host libm (C values down, C values up)
    double *host_lg = nullptr;
    if (exact_host && C > 0) {
        std::vector<u32> hq0(C), hq1(C);
        std::vector<u64> hsb(C);
        SWG_CUDA(cudaMemcpyAsync(hq0.data(), cd.qmin, sizeof(u32) * (size_t)C, cudaMemcpyDeviceToHost, st));
        SWG_CUDA(cudaMemcpyAsync(hq1.data(), cd.qmax, sizeof(u32) * (size_t)C, cudaMemcpyDeviceToHost, st));
        SWG_CUDA(cudaMemcpyAsync(hsb.data(), cd.sum_block, sizeof(u64) * (size_t)C, cudaMemcpyDeviceToHost, st));
        SWG_CUDA(cudaStreamSynchronize(st));
        std::vector<double> lg(C);
        for (u32 ci = 0; ci < C; ci++) {
            const u64 total = (u64)(hq1[ci] - hq0[ci]);
            const u64 gap = total > hsb[ci] ? total - hsb[ci] : 0;
            lg[ci] = gap > 0 ? std::max(std::log((double)gap), 0.0) : 0.0; // paf_filter.rs:902-906
        }
        host_lg = A.take<double>(C);
        SWG_CUDA(cudaMemcpyAsync(host_lg, lg.data(), sizeof(double) * (size_t)C, cudaMemcpyHostToDevice, st));
        SWG_CUDA(cudaStreamSynchronize(st)); // lg lives on this stack frame
    }
    const int nb = bits_for(in.n);
    if (2 * nb > 63) throw RangeError{"too many records for the chain order key"};
    u64 *okey_all = A.take<u64>(C);
    {
        const u64 min_len = cfg.min_scaffold_length;
        const double min_sid = cfg.min_scaffold_identity;
        const u32 seqmask = (u32)((1ull << sb) - 1);
        u64 *hk = P.hk;
        u32 *hv = P.hv;
        const u32 hmask = P.hmask;
        launch_for<t_chain_order>(C, st, lc, [=] __device__(u32 ci) {
            const u32 p = head_pos[ci];
            u64 k = skey[p] >> gshift;
            u8 fwd = (k & 1) == 0;
            u32 tid = (u32)(k >> 1) & seqmask, qid = (u32)(k >> (1 + sb)) & seqmask;
            u32 qmin = cd.qmin[ci], qmax = cd.qmax[ci], tmin = cd.tmin[ci], tmax = cd.tmax[ci];
            u64 sm = cd.sum_matches[ci], sbk = cd.sum_block[ci];
            u64 total = (u64)(qmax - qmin);                         // paf_filter.rs:896
            double wid = chain_identity_fn(total, sbk, sm, cuda_log, host_lg ? host_lg + ci : nullptr); // :901-913
            bool pass = total >= min_len && wid >= min_sid;         // :449-455
            ct.qid[ci] = qid; ct.tid[ci] = tid; ct.fwd[ci] = fwd;
            ct.wid[ci] = wid; ct.pass[ci] = pass ? 1 : 0; // ct.qs / qe / ts / te already hold the bounding box
            bool zero = false;
            if (pass) {
                u32 Aidx = hash_lookup(hk, hv, hmask, ((u64)in.P[qid] << 32) | in.P[tid]);
                okey_all[ci] = ((u64)Aidx << nb) | grp_minidx[gid[p]];
                zero = qmax == qmin || tmax == tmin;
            }
            u32 am = __activemask();
            u32 nz = __popc(__ballot_sync(am, zero));
            if (nz && (threadIdx.x & 31) == (u32)(__ffs(am) - 1)) atomicAdd((unsigned long long *)&ctr[C_PASS_ZEROSPAN], (unsigned long long)nz);
        });
    }
    // only the chains that pass the mass/identity filter take part in the ordering
    u64 *okey = A.take<u64>(C), *okey2 = A.take<u64>(C);
    u32 *oval = A.take<u32>(C), *oval2 = A.take<u32>(C);
    u32 *bsum = A.take<u32>(scan_temp_u32(C));
    scan_flags([=] __device__(u32 ci) -> u32 { return ct.pass[ci] ? 1u : 0u; },
               [=] __device__(u32 ci, u32 ex, u32 v) { if (v) { okey[ex] = okey_all[ci]; oval[ex] = ci; } }, C, bsum, d_cnt + 1, st, lc);
    u32 C1;
    {   // the count and the counters in one round trip
        u32 *h = reinterpret_cast<u32 *>(c->h_ctr + C_COUNT);
        SWG_CUDA(cudaMemcpyAsync(h, d_cnt + 1, sizeof(u32), cudaMemcpyDeviceToHost, st));
        read_counters(c);
        C1 = *h;
    }
    sort_pairs(c, okey, okey2, oval, oval2, C1, 2 * nb); // stable: ties (same group) keep head-position order
    S.n_chains_after_mass = C1;
    return Chains{chain_of, ct, C, C1, okey, oval, c->h_ctr[C_PASS_ZEROSPAN]};
}

// ---- O* + GS: t-space = passing chains in the reference's `filtered_chains` order, scaffold sweep, final order ------------
struct KeptChains {
    u32 C2 = 0;                   // kept chains, numbered u + 1 = 1 .. C2 in chain_N order
    const u32 *fin_t = nullptr;   // fin_t[u] = t of the chain numbered u + 1
    const u32 *t_qs = nullptr, *t_qe = nullptr, *t_ts = nullptr; // t-space columns (t = rank among the passing chains)
    const u64 *t_c2key = nullptr; // chromosome pair
    const u8 *t_fwd = nullptr;
};
static KeptChains order_chains(swg_ctx *c, const swg_config &cfg, const DevIn &in, const Prefiltered &P, const Chains &chains, bool exact_host,
                                swg_stats &S) {
    cudaStream_t st = c->stream; LaunchCounter &lc = c->lc; Arena &A = c->arena;
    const bool cuda_log = c->knobs.cuda_log;
    u64 *ctr = c->d_ctr;
    const u32 C1 = chains.C1;
    const ChainTable ct = chains.ct;
    const int sb = P.sb, nb = bits_for(in.n);
    stage_mark(c, "chain_order");
    if (C1 == 0) return KeptChains{};
    // oc_chain[t] = dense chain id of the t-th filtered chain
    const u32 *oc_chain = chains.oval;
    u32 *t_qs = A.take<u32>(C1), *t_qe = A.take<u32>(C1), *t_ts = A.take<u32>(C1), *t_te = A.take<u32>(C1);
    u64 *t_c2key = A.take<u64>(C1);
    u64 *t_g2key = A.take<u64>(C1);
    u8 *t_fwd = A.take<u8>(C1);
    double *t_score = A.take<double>(C1);
    const int scoring = cfg.scoring_function;
    // first appearance (smallest t) of every chromosome pair and genome pair among the filtered chains: two open-addressing
    // tables with atomicMin (one insert per chain; round 1 sorted the chains twice for this)
    u64 *hk2, *hk3;
    u32 *hv2, *hv3;
    const u32 hmask2 = first_index_table(c, C1, hk2, hv2);
    first_index_table(c, C1, hk3, hv3);
    launch_for<t_tspace>(C1, st, lc, [=] __device__(u32 t) {
        u32 ci = oc_chain[t];
        u32 q = ct.qid[ci], tt = ct.tid[ci];
        t_qs[t] = ct.qs[ci]; t_qe[t] = ct.qe[ci]; t_ts[t] = ct.ts[ci]; t_te[t] = ct.te[ci];
        const u64 c2 = ((u64)q << sb) | tt, g2 = ((u64)in.P2[q] << sb) | in.P2[tt];
        t_c2key[t] = c2;
        t_g2key[t] = g2;
        t_fwd[t] = ct.fwd[ci];
        t_score[t] = score_fn(scoring, ct.wid[ci], ct.qs[ci], ct.qe[ci], cuda_log);
        hash_insert_min(hk2, hv2, hmask2, c2, t);
        hash_insert_min(hk3, hv3, hmask2, g2, t);
    });
    if (exact_host) { // exact re-rank: the chain scores from the host libm as well
        std::vector<double> hw(C1), hs(C1);
        std::vector<u32> hq0(C1), hq1(C1);
        double *d_w = A.take<double>(C1);
        launch_for<t_tspace>(C1, st, lc, [=] __device__(u32 t) { d_w[t] = ct.wid[oc_chain[t]]; });
        SWG_CUDA(cudaMemcpyAsync(hw.data(), d_w, sizeof(double) * (size_t)C1, cudaMemcpyDeviceToHost, st));
        SWG_CUDA(cudaMemcpyAsync(hq0.data(), t_qs, sizeof(u32) * (size_t)C1, cudaMemcpyDeviceToHost, st));
        SWG_CUDA(cudaMemcpyAsync(hq1.data(), t_qe, sizeof(u32) * (size_t)C1, cudaMemcpyDeviceToHost, st));
        SWG_CUDA(cudaStreamSynchronize(st));
        for (u32 t = 0; t < C1; t++) hs[t] = host_score(scoring, hw[t], hq0[t], hq1[t]);
        SWG_CUDA(cudaMemcpyAsync(t_score, hs.data(), sizeof(double) * (size_t)C1, cudaMemcpyHostToDevice, st));
        SWG_CUDA(cudaStreamSynchronize(st)); // hs lives on this stack frame
    }
    u32 *g2min = A.take<u32>(C1);
    u64 *sk = A.take<u64>(C1), *sk2 = A.take<u64>(C1);
    u32 *sv = A.take<u32>(C1), *sv2 = A.take<u32>(C1);
    // scaffold plane sweep (plane_sweep_scaffold.rs:47-251)
    u8 *t_keep = nullptr;
    u64 nq, nt;
    if (cfg.scaffold_filter_mode == SWG_ONE_TO_ONE) { nq = 1; nt = 1; }
    else { nq = cfg.scaffold_max_per_query; nt = cfg.scaffold_max_per_target; }
    const bool need_sweep = C1 > 1 && (nq != SWG_KEEP_ALL || nt != SWG_KEEP_ALL || chains.pass_zero > 0);
    if (need_sweep) {
        u8 *k1 = A.take<u8>(C1);
        t_keep = A.take<u8>(C1);
        general_sweep(c, C1, nullptr, 0, t_c2key, 2 * sb, P.cb, t_qs, t_qe, t_score, nq, cfg.scaffold_overlap_threshold, k1);
        general_sweep(c, C1, k1, 1, t_c2key, 2 * sb, P.cb, t_ts, t_te, t_score, nt, cfg.scaffold_overlap_threshold, t_keep);
    }
    // final order: (g2min, c2min, t) in ONE stable sort (t is the input order); dropped chains sort last
    const int ob = bits_for(C1);
    if (2 * ob + 1 > 64) throw RangeError{"too many chains for the final order key"};
    {
        u64 *skw = sk;
        u32 *svw = sv;
        launch_for<t_keys_g2min>(C1, st, lc, [=] __device__(u32 t) {
            const bool kept = t_keep ? t_keep[t] != 0 : true;
            const u32 gm = hash_lookup(hk3, hv3, hmask2, t_g2key[t]), cm = hash_lookup(hk2, hv2, hmask2, t_c2key[t]);
            g2min[t] = gm;
            skw[t] = kept ? (((u64)gm << ob) | cm) : (1ull << (2 * ob));
            svw[t] = t;
            const u32 am = __activemask();
            const u32 nk = __popc(__ballot_sync(am, kept));
            if (nk && (threadIdx.x & 31) == (u32)(__ffs(am) - 1)) atomicAdd((unsigned long long *)&ctr[C_KEPT_CHAINS], (unsigned long long)nk);
        });
    }
    read_counters_begin(c); // the kept-chain count is final here; the host picks it up while the sort runs
    sort_pairs(c, sk, sk2, sv, sv2, C1, 2 * ob + 1);
    read_counters_end(c);
    const u32 C2 = (u32)c->h_ctr[C_KEPT_CHAINS];
    S.score_near_ties = c->h_ctr[C_NEAR_TIES];
    {
        const u32 *fin = sv;
        // chain number + the order key of its genome-pair group (first-appearance indices A, B of the group's first
        // filtered chain): what a multi-GPU driver needs to merge the per-shard numberings (swg_last_chain_keys)
        c->keys.reserve(((size_t)C2 + 1) * 8 + 1024); // context-owned: later calls that rewind the scratch arena do not touch it
        u32 *keyA = c->keys.take<u32>(C2 + 1), *keyB = c->keys.take<u32>(C2 + 1);
        const u64 *okc = chains.okey;
        const u64 bmask = (1ull << nb) - 1;
        launch_for<t_final_k>(C2, st, lc, [=] __device__(u32 u) {
            const u32 t = fin[u];
            ct.k[oc_chain[t]] = u + 1;
            const u64 gk = okc[g2min[t]];
            keyA[u] = (u32)(gk >> nb);
            keyB[u] = (u32)(gk & bmask);
        });
        c->last_keyA = keyA;
        c->last_keyB = keyB;
    }
    c->last_n_chains = C2;
    S.n_chains_kept = C2;
    return KeptChains{C2, sv, t_qs, t_qe, t_ts, t_c2key, t_fwd};
}

// ---- K5: anchors = members of kept chains (paf_filter.rs:517-528) ---------------------------------
// One thread per four sorted positions (striped over a 1024-position block).  Counts the anchors it writes into C_ANCHORS, one
// atomic per block.  EMIT: also appends the inversion candidates (alive, reverse strand, not an anchor) to inv_list in no
// particular order, one atomic on *inv_n per block.  That list equals the flag scan over all N records only when every alive
// record is a sorted position (n_m == n_alive).
template <bool EMIT>
__global__ void __launch_bounds__(256) k_assign(u32 n_m, const u32 *__restrict__ chain_of, SortedIdx sidx, ChainTable ct, u8 *flags,
                                                u8 *__restrict__ status, u32 *__restrict__ chain_id, u64 *ctr, u32 *__restrict__ inv_list,
                                                u32 *inv_n) {
    __shared__ u32 s_w[8][4];
    __shared__ u32 s_base;
    const u32 lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const u32 base = blockIdx.x * 1024;
    u32 rec[4], m[4], n_anchor = 0;
    bool cand[4];
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const u32 p = base + k * 256 + threadIdx.x;
        cand[k] = false;
        rec[k] = 0;
        if (p < n_m) {
            const u32 ci = chain_of[p];
            const u32 i = sidx[p];
            const u32 kk = ct.k[ci];
            if (kk) { status[i] = 1; chain_id[i] = kk; n_anchor++; }
            const u8 add = (u8)((kk ? F_ANCHOR : 0) | (ct.pass[ci] ? F_PREMEM : 0));
            if (EMIT) {
                const u8 fl = flags[i];
                cand[k] = !kk && (fl & (F_ALIVE | F_REV)) == (F_ALIVE | F_REV);
                if (add) flags[i] = fl | add;
            } else if (add) flags[i] |= add;
            rec[k] = i;
        }
        if (EMIT) {
            m[k] = __ballot_sync(0xFFFFFFFFu, cand[k]);
            if (lane == 0) s_w[warp][k] = __popc(m[k]);
        }
    }
    const int slots[1] = {C_ANCHORS};
    const u32 vals[1] = {n_anchor};
    block_count_add<1>(ctr, slots, vals); // (its barriers also publish s_w)
    if (!EMIT) return;
    if (threadIdx.x == 0) {
        u32 tot = 0;
        for (int k = 0; k < 4; k++)
            for (int w = 0; w < 8; w++) { const u32 t = s_w[w][k]; s_w[w][k] = tot; tot += t; }
        s_base = tot ? atomicAdd(inv_n, tot) : 0;
    }
    __syncthreads();
    const u32 lt = lanemask_lt();
#pragma unroll
    for (int k = 0; k < 4; k++)
        if (cand[k]) inv_list[s_base + s_w[warp][k] + __popc(m[k] & lt)] = rec[k];
}

// The inversion candidates of the default path, emitted by the anchor pass (k_assign<true>); nullptr list: capture_inversions
// compacts them itself with a flag scan over all records.
struct InvCands { u32 *list = nullptr, *n = nullptr; };

// inversion capture through the buckets of inversion_grid: a huge group (or SWG_INV_GRID=1), when its key fits 64 bits.  wb0 is the
// widest query bucket: 2^wb0 > 2 * jump.
static int inversion_grid_wb0(const swg_config &cfg) { return std::max(17, bits_for(2 * cfg.scaffold_gap + 1)); }
static bool takes_inversion_grid(const swg_ctx *c, const swg_config &cfg, const Prefiltered &P, u32 n_huge) {
    const int wb0 = inversion_grid_wb0(cfg);
    return (n_huge > 0 || c->knobs.inv_grid) && 2 * P.sb + (P.cb > wb0 ? P.cb - wb0 : 1) + 1 <= 64;
}

static InvCands assign_anchors(swg_ctx *c, const Ordered &O, const Chains &chains, u8 *flags, u8 *status, u32 *chain_id, bool emit_candidates) {
    const u32 n_m = O.n_m;
    InvCands inv;
    if (emit_candidates) {
        inv.list = c->arena.take<u32>(n_m);
        inv.n = c->arena.take<u32>(1);
        SWG_CUDA(cudaMemsetAsync(inv.n, 0, sizeof(u32), c->stream));
        k_assign<true><<<cdiv(n_m, 1024), 256, 0, c->stream>>>(n_m, chains.chain_of, O.sidx, chains.ct, flags, status, chain_id, c->d_ctr,
                                                             inv.list, inv.n);
    } else {
        k_assign<false><<<cdiv(n_m, 1024), 256, 0, c->stream>>>(n_m, chains.chain_of, O.sidx, chains.ct, flags, status, chain_id, c->d_ctr,
                                                              nullptr, nullptr);
    }
    c->lc.n++;
    return inv;
}

// ---- K6: inversion capture (paf_filter.rs:535-597) ------------------------------------------------
// Does a reverse mapping (query interval [mqs, mqe], centres qc / tc) belong to the '+' chain that starts at (cqs, cts) and ends at
// query cqe?  Its query interval must touch the chain's, extended by G on both sides, and its centre must lie within
// floor(|dev| / sqrt 2) <= G of the chain's diagonal.
static __device__ __forceinline__ bool inversion_hit(u64 mqs, u64 mqe, u64 qc, u64 tc, u64 cqs, u64 cqe, u64 cts, u64 G) {
    const u64 ext_s = cqs > G ? cqs - G : 0, ext_e = cqe + G;
    if (mqe < ext_s || mqs > ext_e) return false;
    const i64 dv = (i64)tc - (i64)qc - ((i64)cts - (i64)cqs);
    const u64 dev = dv < 0 ? (u64)(-dv) : (u64)dv;
    return (u64)__ddiv_rn((double)dev, 1.4142135623730951) <= G;
}

// A chromosome pair that holds a huge group can hold 10^5..10^6 kept chains; walking all of them for every reverse mapping is
// O(n * chains).  Then chains and mappings meet in buckets of the query axis (2^wb0: the widest bucket) and of the diagonal.
// ik[u] = chromosome pair of the kept chain u if it is a '+' chain, NONE64 for a '-' chain; u_qs / u_qe / u_ts its coordinates.
static void inversion_grid(swg_ctx *c, const swg_config &cfg, const DevIn &in, const Prefiltered &P, u32 C2, const u64 *ik, const u32 *u_qs,
                           const u32 *u_qe, const u32 *u_ts, int wb0, u8 *status, u32 *chain_id) {
    cudaStream_t st = c->stream; LaunchCounter &lc = c->lc; Arena &A = c->arena;
    const Knobs &K = c->knobs;
    const u32 N = in.n;
    u8 *flags = P.flags;
    u64 *ctr = c->d_ctr;
    const int sb = P.sb, cb = P.cb;
    stage_mark(c, "inversion_grid");
    const u64 G = cfg.scaffold_gap;
    const u64 maxc = P.maxcoord;
    u32 *d_cnt = A.take<u32>(2); // [0] entries, [1] candidate mappings
    u32 *inv_list = A.take<u32>(N);
    u32 *bsum = A.take<u32>(scan_temp_u32(N));
    scan_flags([=] __device__(u32 i) -> u32 { return (flags[i] & (F_ALIVE | F_REV | F_ANCHOR)) == (F_ALIVE | F_REV) ? 1u : 0u; },
               [=] __device__(u32 i, u32 ex, u32 v) { if (v) inv_list[ex] = i; }, N, bsum, d_cnt + 1, st, lc);
    // Bucket width of the query axis.  The chains of a (pair, '+') group are numbered in query order, so the entries of a bucket
    // ascend along the query axis and a mapping in the middle of a wide bucket walks every chain that ends more than a jump to
    // its left before the first it can belong to (20 M pile, 2^17: 1560 entries per mapping).  Narrow buckets make nearly every
    // entry of a cell a hit on the query axis; they cost entries (a chain enters every bucket its extended interval touches)
    // and cells per mapping.  Both are counted for the widths 2^wb0 .. 2^12 and the narrowest width within budget is taken.
    constexpr int NW = 6;
    unsigned long long *wcnt = (unsigned long long *)A.take<u64>(2 * NW);
    SWG_CUDA(cudaMemsetAsync(wcnt, 0, 2 * NW * sizeof(u64), st));
    launch_for<t_invw>(C2, st, lc, [=] __device__(u32 u) {
        const bool f = ik[u] != NONE64;
        const u64 a0 = u_qs[u] > G ? (u64)u_qs[u] - G : 0, e0 = (u64)u_qe[u] + G < maxc ? (u64)u_qe[u] + G : maxc;
        const u32 am = __activemask();
#pragma unroll
        for (int k = 0; k < NW; k++) {
            const int w = wb0 - k;
            const u32 v = f && w >= 12 ? (u32)((e0 >> w) - (a0 >> w) + 1) : 0u;
            const u32 sum = __reduce_add_sync(am, v);
            if (sum && (threadIdx.x & 31) == (u32)(__ffs(am) - 1)) atomicAdd(&wcnt[k], (unsigned long long)sum);
        }
    });
    launch_for_dev<t_invw2>(d_cnt + 1, c->sm_count, st, lc, [=] __device__(u32 x) {
        const u32 i = inv_list[x];
        const u64 qs0 = in.qs[i], qe0 = in.qe[i];
        const u32 am = __activemask();
#pragma unroll
        for (int k = 0; k < NW; k++) {
            const int w = wb0 - k;
            const u32 v = w >= 12 ? (u32)((qe0 >> w) - (qs0 >> w) + 1) : 0u;
            const u32 sum = __reduce_add_sync(am, v);
            if (sum && (threadIdx.x & 31) == (u32)(__ffs(am) - 1)) atomicAdd(&wcnt[NW + k], (unsigned long long)sum);
        }
    });
    u32 *h2 = reinterpret_cast<u32 *>(c->h_ctr + C_COUNT);
    unsigned long long hw[2 * NW];
    SWG_CUDA(cudaMemcpyAsync(h2 + 1, d_cnt + 1, sizeof(u32), cudaMemcpyDeviceToHost, st));
    SWG_CUDA(cudaMemcpyAsync(hw, wcnt, sizeof hw, cudaMemcpyDeviceToHost, st));
    SWG_CUDA(cudaStreamSynchronize(st));
    int wb = wb0;
    // (only where chains are many: a pair with a pile holds 10^5 and more; a few hundred chromosome-scale chains would just be cut
    // into thousands of entries each)
    for (int k = NW - 1; k > 0; k--) {
        const int w = wb0 - k;
        if (w < 12 || K.inv_wide || (C2 < 65536 && !K.inv_narrow)) continue;
        const bool fits = 2 * sb + (cb > w ? cb - w : 1) + 1 <= 64;
        if (fits && hw[k] <= std::max<u64>(1ull << 25, 8ull * C2) && hw[k] < (1ull << 31) && hw[NW + k] <= 3ull * h2[1] + 1024) { wb = w; break; }
    }
    const int bb = cb > wb ? cb - wb : 1;
    // ... and in buckets of the diagonal (target_start - query_start of a chain against the centre diagonal of a mapping): the
    // deviation test floor(|dev| / sqrt 2) <= G admits |dev| <= R only, so a mapping meets the chains of the diagonal buckets
    // that [dm - R, dm + R] touches.  Width: an eighth of 2 R + 1 (a mapping walks up to ten narrow cells, but a cell it can only
    // fail in is small); wider while the key would pass 64 bits, no diagonal buckets if it still does.
    const u64 R = (u64)std::ceil((double)(G + 1) * 1.4142135623730951) + 1; // |dev| > R  =>  perp > G
    int wd = std::max(bits_for(2 * R + 1) - 3, 8);
    const u64 doff = maxc + 1; // diagonals are shifted to be non-negative: they lie in [-maxc, maxc]
    int db = bits_for((2 * maxc + 2) >> wd);
    while (2 * sb + bb + db > 64 && wd < bits_for(2 * R + 1)) { wd++; db = bits_for((2 * maxc + 2) >> wd); }
    if (2 * sb + bb + db > 64 || K.inv_no_diag) db = 0;
    // entries: every kept '+' chain once per bucket its extended query interval [qs - G, qe + G] touches
    u32 *e_off = A.take<u32>(C2);
    auto first_b = [=] __device__(u32 u) -> u32 { const u64 a = u_qs[u]; return (u32)((a > G ? a - G : 0) >> wb); };
    auto last_b = [=] __device__(u32 u) -> u32 { const u64 e = (u64)u_qe[u] + G; return (u32)((e < maxc ? e : maxc) >> wb); };
    scan_apply([=] __device__(u32 u) -> u32 { return ik[u] != NONE64 ? last_b(u) - first_b(u) + 1 : 0u; },
               [=] __device__(u32 u, u32 ex, u32) { e_off[u] = ex; }, C2, bsum, d_cnt, st, lc);
    SWG_CUDA(cudaMemcpyAsync(h2, d_cnt, sizeof(u32), cudaMemcpyDeviceToHost, st));
    SWG_CUDA(cudaStreamSynchronize(st));
    const bool dbg = K.stage_timing;
    if (dbg) fprintf(stderr, "[swg inversion] query buckets 2^%d (widest 2^%d), diagonal buckets 2^%d (%d bits)\n", wb, wb0, wd, db);
    const u32 n_ent = h2[0], n_inv = h2[1];
    if (!n_ent || !n_inv) return;
    u64 *ek = A.take<u64>(n_ent), *ek2 = A.take<u64>(n_ent);
    u32 *ev = A.take<u32>(n_ent), *ev2 = A.take<u32>(n_ent);
    launch_for<t_invent>(C2, st, lc, [=] __device__(u32 u) {
        if (ik[u] == NONE64) return;
        const u32 b0 = first_b(u), b1 = last_b(u);
        u32 o = e_off[u];
        const u64 dg = db ? ((u64)((i64)u_ts[u] - (i64)u_qs[u] + (i64)doff) >> wd) : 0;
        for (u32 b = b0; b <= b1; b++, o++) { ek[o] = (((ik[u] << bb) | b) << db) | dg; ev[o] = u; }
    });
    sort_pairs(c, ek, ek2, ev, ev2, n_ent, 2 * sb + bb + db); // stable: chains stay in k order inside a bucket
    uint4 *ent = A.take<uint4>(n_ent);
    {
        const u32 *evc = ev;
        launch_for<t_gather>(n_ent, st, lc, [=] __device__(u32 x) { const u32 u = evc[x]; ent[x] = make_uint4(u_qs[u], u_qe[u], u_ts[u], u); });
    }
    // the candidates ordered by (pair, first bucket): neighbouring threads walk the same entries
    u64 *qk = A.take<u64>(n_inv), *qk2 = A.take<u64>(n_inv);
    u32 *qv = A.take<u32>(n_inv), *qv2 = A.take<u32>(n_inv);
    launch_for<t_invkeys>(n_inv, st, lc, [=] __device__(u32 x) {
        const u32 i = inv_list[x];
        qk[x] = (((((u64)in.qid[i] << sb) | in.tid[i])) << bb) | ((u64)in.qs[i] >> wb);
        qv[x] = i;
    });
    sort_pairs(c, qk, qk2, qv, qv2, n_inv, 2 * sb + bb);
    const u64 *ekc = ek, *qkc = qk;
    const u32 *qvc = qv;
    unsigned long long *inv_dbg = (unsigned long long *)A.take<u64>(4);
    SWG_CUDA(cudaMemsetAsync(inv_dbg, 0, 4 * sizeof(u64), st));
    launch_for<t_inversion>(n_inv, st, lc, [=] __device__(u32 x0) {
        u32 n_walk = 0, n_cells = 0;
        const u32 i = qvc[x0];
        const u64 mqs = in.qs[i], mqe = in.qe[i], mts = in.ts[i], mte = in.te[i];
        const u64 qc = (mqs + mqe) / 2, tc = (mts + mte) / 2;
        const u64 pairkey = qkc[x0] >> bb;
        u32 best = NONE32; // smallest u = the first chain in the reference's order (paf_filter.rs:553-596)
        const u64 dm = (u64)((i64)tc - (i64)qc + (i64)doff);
        const u64 d0 = db ? (dm > R ? dm - R : 0) >> wd : 0, d1 = db ? (dm + R) >> wd : 0;
        for (u64 b = mqs >> wb; b <= (mqe >> wb); b++)
        for (u64 dg = d0; dg <= d1; dg++) {
            const u64 key = (((pairkey << bb) | b) << db) | dg;
            u32 lo = 0, hi = n_ent;
            while (lo < hi) { const u32 mid = (lo + hi) >> 1; if (ekc[mid] < key) lo = mid + 1; else hi = mid; }
            n_cells++;
            for (u32 x = lo; x < n_ent && ekc[x] == key; x++) {
                n_walk++;
                const uint4 ch = ent[x];
                if (ch.w >= best) break; // entries of a bucket ascend in u
                if (inversion_hit(mqs, mqe, qc, tc, ch.x, ch.y, ch.z, G)) { best = ch.w; break; }
            }
        }
        if (best != NONE32) { status[i] = 1; chain_id[i] = best + 1; flags[i] |= F_ANCHOR; }
        warp_count_add(ctr, C_ANCHORS, best != NONE32);
        if (dbg) { atomicAdd(&inv_dbg[0], (unsigned long long)n_walk); atomicAdd(&inv_dbg[1], (unsigned long long)n_cells); atomicMax(&inv_dbg[2], (unsigned long long)n_walk); if (best != NONE32) atomicAdd(&inv_dbg[3], 1ull); }
    });
    if (dbg) {
        unsigned long long hd[4];
        SWG_CUDA(cudaMemcpyAsync(hd, inv_dbg, sizeof hd, cudaMemcpyDeviceToHost, st));
        SWG_CUDA(cudaStreamSynchronize(st));
        fprintf(stderr, "[swg inversion] %u candidates, %u entries, %llu entries walked (max %llu per candidate), %llu cells, %llu captured\n", n_inv, n_ent, hd[0], hd[2], hd[1], hd[3]);
    }
}

// kept chains in chain_N order u; ik[u] = chromosome pair of a '+' chain, NONE64 for a '-' chain; u_c2[u] = the pair of either.  The
// final order groups the chains by chromosome pair, so a pair's chains are one run of u: the table below maps a pair to the start
// of its run (atomicMin of u).
static void capture_inversions(swg_ctx *c, const swg_config &cfg, const DevIn &in, const Prefiltered &P, u32 n_huge, const KeptChains &kc,
                               const InvCands &cands, u8 *status, u32 *chain_id) {
    cudaStream_t st = c->stream; LaunchCounter &lc = c->lc; Arena &A = c->arena;
    const u32 N = in.n, C2 = kc.C2;
    u8 *flags = P.flags;
    u64 *ctr = c->d_ctr;
    const int sb = P.sb;
    const u32 *t_qs = kc.t_qs, *t_qe = kc.t_qe, *t_ts = kc.t_ts;
    const u64 *t_c2key = kc.t_c2key;
    const u8 *t_fwd = kc.t_fwd;
    u64 *ik = A.take<u64>(C2), *ik2 = A.take<u64>(C2);
    u32 *iv = A.take<u32>(C2), *iv2 = A.take<u32>(C2);
    u32 *u_qs = A.take<u32>(C2), *u_qe = A.take<u32>(C2), *u_ts = A.take<u32>(C2);
    u64 *u_c2 = A.take<u64>(C2);
    u64 *hk4;
    u32 *hv4;
    const u32 hmask4 = first_index_table(c, C2, hk4, hv4);
    {
        const u32 *fin = kc.fin_t;
        launch_for<t_invkeys>(C2, st, lc, [=] __device__(u32 u) {
            u32 t = fin[u];
            bool f = t_fwd[t] != 0;
            const u64 c2 = t_c2key[t];
            ik[u] = f ? c2 : NONE64;
            iv[u] = u;
            u_c2[u] = c2;
            u_qs[u] = t_qs[t]; u_qe[u] = t_qe[t]; u_ts[u] = t_ts[t];
            hash_insert_min(hk4, hv4, hmask4, c2, u);
        });
    }
    if (takes_inversion_grid(c, cfg, P, n_huge)) {
        inversion_grid(c, cfg, in, P, C2, ik, u_qs, u_qe, u_ts, inversion_grid_wb0(cfg), status, chain_id);
        return;
    }
    // the candidates (reverse strand, alive, not yet an anchor: a few per cent of the records) come as a list in no particular
    // order (each is judged on its own): from the anchor pass, else compacted here; a candidate looks its chromosome pair up
    // and walks the pair's run of chains in chain_N order — the reference's loop over the kept '+' chains "in order", first
    // hit wins (paf_filter.rs:553-596)
    const u64 G = cfg.scaffold_gap;
    const u64 *ikc = ik;
    u32 *inv_list = cands.list, *d_ninv = cands.n;
    if (!inv_list) {
        inv_list = A.take<u32>(N);
        d_ninv = A.take<u32>(1);
        u32 *bsum = A.take<u32>(scan_temp_u32(N));
        scan_flags([=] __device__(u32 i) -> bool { return (flags[i] & (F_ALIVE | F_REV | F_ANCHOR)) == (F_ALIVE | F_REV); },
                   [=] __device__(u32 i, u32 slot, u32 v) { if (v) inv_list[slot] = i; }, N, bsum, d_ninv, st, lc);
    }
    launch_for_dev<t_inversion>(d_ninv, c->sm_count, st, lc, [=] __device__(u32 x0) {
        const u32 i = inv_list[x0];
        const u64 key = ((u64)in.qid[i] << sb) | in.tid[i];
        const u32 u0 = hash_lookup(hk4, hv4, hmask4, key);
        bool hit = false;
        if (u0 != NONE32) {
            u64 mqs = in.qs[i], mqe = in.qe[i], mts = in.ts[i], mte = in.te[i];
            u64 qc = (mqs + mqe) / 2, tc = (mts + mte) / 2;
            for (u32 u = u0; u < C2 && u_c2[u] == key; u++) {
                if (ikc[u] == NONE64) continue; // a '-' chain
                if (inversion_hit(mqs, mqe, qc, tc, u_qs[u], u_qe[u], u_ts[u], G)) { status[i] = 1; chain_id[i] = u + 1; flags[i] |= F_ANCHOR; hit = true; break; }
            }
        }
        warp_count_add(ctr, C_ANCHORS, hit);
    });
}

// ---- K7: rescue (paf_filter.rs:613-732) -----------------------------------------------------
static void rescue(swg_ctx *c, const swg_config &cfg, const DevIn &in, const Prefiltered &P, u8 *status, u32 *chain_id) {
    cudaStream_t st = c->stream; LaunchCounter &lc = c->lc; Arena &A = c->arena;
    const Knobs &K = c->knobs;
    const u32 N = in.n;
    u8 *flags = P.flags;
    u64 *ctr = c->d_ctr;
    const int sb = P.sb, cb = P.cb;
    const u64 D = cfg.scaffold_max_deviation;
    // anchor list (status == 1) ordered by (chromosome pair, query center); one sort when the key fits 64 bits,
    // else two chained stable sorts (center first, then the pair)
    const bool wide_a = (2 * sb + cb > 63) || K.force_wide;
    u64 *ak = A.take<u64>(N), *ak2 = A.take<u64>(N);
    u32 *av = A.take<u32>(N), *av2 = A.take<u32>(N);
    u32 *d_na = A.take<u32>(2);
    u32 *bsum = A.take<u32>(scan_temp_u32(N));
    u32 NA = 0;
    u64 *apair = nullptr;
    u32 *aqc = nullptr;
    bool a_done = false;
    const int ibN = bits_for(N - 1);
    if (P.gsort && !wide_a && c->rows_grouped && cb + ibN <= 64 && 2 * sb + 1 + ibN <= 64) {
        // the group sort with the chromosome pair as group (the strand bit of the table index stays 0) and the query centre as
        // secondary key: anchors come grouped like the records and nearly in centre order
        const u32 dead = (1u << (2 * sb + 1)) - 1;
        {
            u64 *kk = ak;
            launch_for<t_anchor_keys>(N, st, lc, [=] __device__(u32 i) {
                const bool anchor = (flags[i] & F_ANCHOR) != 0;
                const u64 qc = ((u64)in.qs[i] + in.qe[i]) / 2;
                kk[i] = anchor ? ((((((u64)in.qid[i] << sb) | in.tid[i]) << 1) << cb) | qc) : (((u64)dead << cb) | ((1ull << cb) - 1));
            });
        }
        aqc = A.take<u32>((size_t)N + 1);
        const GroupSorted gs = group_sort(c, ak, ak2, ak, av2, N, cb, GsIndex{1, sb, in.n_seq}, dead, P.g_entries, ibN, group_sort_limit(K), false, aqc);
        if (gs.done) {
            a_done = true;
            NA = gs.n_rec;
            apair = A.take<u64>((size_t)NA + 1);
            const u64 *w = ak;
            const u64 imask = (1ull << ibN) - 1;
            u64 *ap = apair;
            u32 *avw = av;
            launch_for<t_gather>(NA, st, lc, [=] __device__(u32 x) { ap[x] = w[x] >> (ibN + 1); avw[x] = (u32)(w[x] & imask); });
        }
    }
    if (!a_done) {
        scan_flags([=] __device__(u32 i) -> bool { return (flags[i] & F_ANCHOR) != 0; },
                   [=] __device__(u32 i, u32 ex, u32 v) {
                       if (!v) return;
                       u64 qc = ((u64)in.qs[i] + in.qe[i]) / 2;
                       ak[ex] = wide_a ? qc : (((((u64)in.qid[i] << sb) | in.tid[i]) << cb) | qc);
                       av[ex] = i;
                   },
                   N, bsum, d_na, st, lc);
        NA = read_u32(c, d_na);
        if (!wide_a) sort_pairs(c, ak, ak2, av, av2, NA, 2 * sb + cb);
        else sort_pairs_wide(c, ak, ak2, av, av2, NA, cb, 2 * sb, [=] __device__(u32 i) { return ((u64)in.qid[i] << sb) | in.tid[i]; });
        apair = A.take<u64>(NA + 1);
        aqc = A.take<u32>(NA + 1);
        const u64 *akc = ak;
        const u32 *avc = av;
        const u64 cmask = (1ull << cb) - 1;
        u64 *ap = apair;
        u32 *aq = aqc;
        launch_for<t_anchor_keys>(NA, st, lc, [=] __device__(u32 x) {
            if (wide_a) { const u32 i = avc[x]; ap[x] = akc[x]; aq[x] = (u32)(((u64)in.qs[i] + in.qe[i]) / 2); }
            else { ap[x] = akc[x] >> cb; aq[x] = (u32)(akc[x] & cmask); }
        });
    }
    // candidates (alive, not an anchor, not a member of a swept-away scaffold), compacted so the searches run dense
    u32 *rlist = A.take<u32>(N);
    scan_flags([=] __device__(u32 i) -> bool { return (flags[i] & (F_ALIVE | F_ANCHOR | F_PREMEM)) == F_ALIVE; },
               [=] __device__(u32 i, u32 slot, u32 v) { if (v) rlist[slot] = i; }, N, bsum, d_na + 1, st, lc);
    const u32 *avc = av;
    const u32 *d_nr = d_na + 1;
    // The reference squares in u64 and wraps (a release build): qd^2 + td^2 passes 2^64 once td reaches ~0.866 * 2^32, and the
    // wrapped sum can put a far anchor inside D.  Every scanned anchor has qd <= D and td <= max(tc, maxcoord - tc) (anchor
    // centres lie in [0, maxcoord]), so for a candidate with (D^2 + that^2 < 2^64) the sum never wraps and the two shortcuts
    // below hold; for any other candidate every anchor with qd <= D is measured.  Only target centres beyond 3.7 * 10^9 from
    // one end of the coordinate range take that path (on a repeat pile it costs O(anchors within +-D) per candidate).
    const u64 wrap_lim = ~0ull - D * D; // D < 2^31 (checked on entry)
    const bool may_wrap = (u64)P.maxcoord * P.maxcoord > wrap_lim;
    const u64 maxc = P.maxcoord;
    launch_for_dev<t_rescue>(d_nr, c->sm_count, st, lc, [=] __device__(u32 x0) {
        const u32 i = rlist[x0];
        const u64 pair = ((u64)in.qid[i] << sb) | in.tid[i];
        const u64 qc = ((u64)in.qs[i] + in.qe[i]) / 2, tc = ((u64)in.ts[i] + in.te[i]) / 2;
        const u64 td_max = tc > maxc - tc ? tc : maxc - tc;
        const bool wrap = may_wrap && td_max * td_max > wrap_lim;
        // first anchor of the pair at or right of the query center; the scan runs outwards from there and stops once
        // the query-axis distance alone exceeds the best distance found: dist = floor(sqrt(qd^2 + td^2)) >= qd - 1 (the f64
        // square root of a rounded sum can fall one short), so nothing beyond qd > best + 1 can win or tie.  On a repeat pile
        // (10^5..10^6 anchors inside +-D) that is a handful of anchors instead of all of them.  Not when the sum may wrap.
        u32 lo = 0, hi = NA;
        while (lo < hi) {
            u32 mid = (lo + hi) >> 1;
            const u64 mp = apair[mid];
            if (mp < pair || (mp == pair && (u64)aqc[mid] < qc)) lo = mid + 1; else hi = mid;
        }
        u64 best_d = NONE64;
        u32 best_a = NONE32;
        auto visit = [&](u32 x, u64 qd) {
            const u32 a = avc[x];
            const u64 atc = ((u64)in.ts[a] + in.te[a]) / 2;
            const u64 td = atc > tc ? atc - tc : tc - atc;
            if (td > D && !wrap) return; // then floor(sqrt(qd^2+td^2)) > D
            const u64 dist = (u64)__dsqrt_rn((double)(qd * qd + td * td)); // u64: wraps like the reference
            if (dist <= D && (dist < best_d || (dist == best_d && a < best_a))) { best_d = dist; best_a = a; }
        };
        for (u32 x = lo; x < NA && apair[x] == pair; x++) {
            const u64 qd = (u64)aqc[x] - qc;
            if (qd > D || (!wrap && best_a != NONE32 && qd > best_d + 1)) break;
            visit(x, qd);
        }
        for (u32 x = lo; x > 0;) {
            x--;
            if (apair[x] != pair) break;
            const u64 qd = qc - (u64)aqc[x];
            if (qd > D || (!wrap && best_a != NONE32 && qd > best_d + 1)) break;
            visit(x, qd);
        }
        if (best_a != NONE32) { status[i] = 2; chain_id[i] = chain_id[best_a]; }
        warp_count_add(ctr, C_RESCUED, best_a != NONE32);
    });
}

// exact_host: every logarithm on the path comes from the HOST libm (in.score carries the record scores; the chain-level
// logs are computed on the host from small downloads) — the exact re-rank of DESIGN 4d, not the normal path.
static void run_filter(swg_ctx *c, const swg_config &cfg, const DevIn &in, u8 *status, u32 *chain_id, swg_stats *stats,
                       cudaEvent_t ev_matches = nullptr /* recorded when in.matches has arrived (swg_filter overlaps that copy) */,
                       bool exact_host = false) {
    const u32 N = in.n;
    const u64 launches0 = c->lc.n;
    swg_stats S;
    std::memset(&S, 0, sizeof S);
    S.n_input = N;
    c->sort_passes = 0;
    c->sort_pairs = 0;
    c->sort_bytes_per_pair = 24;
    c->stage_used = 0;
    c->last_n_chains = 0;
    c->last_keyA = c->last_keyB = nullptr;
    c->last_flags = nullptr;
    if (N == 0) { SWG_CUDA(cudaStreamSynchronize(c->stream)); finish(c, S, launches0, stats); return; }
    // (status / chain_id are cleared by prefilter, while the host waits for the first small read)
    if (cfg.scaffold_gap >= (1ull << 31) || cfg.scaffold_max_deviation >= (1ull << 31))
        throw RangeError{"scaffold_gap / scaffold_max_deviation must be < 2^31"};

    const Limits lim = mapping_limits(cfg);
    const Prefiltered P = prefilter(c, cfg, in, lim, status, chain_id, ev_matches, S);
    const Kept kept = primary_sweep(c, cfg, in, P, lim, ev_matches);
    if (cfg.scaffold_gap == 0) { // no-scaffold exit (paf_filter.rs:409-434)
        k_unassigned<<<cdiv(N, 256), 256, 0, c->stream>>>(N, P.flags, kept.q, kept.t, status, c->d_ctr);
        c->lc.n++;
        read_counters(c);
        S.n_after_sweep = S.n_kept = c->h_ctr[C_KEPT];
        S.score_near_ties = c->h_ctr[C_NEAR_TIES];
        finish(c, S, launches0, stats);
        return;
    }
    const Ordered O = order_records(c, cfg, in, P, kept, S);
    if (O.n_m == 0) { finish(c, S, launches0, stats); return; }
    const Chained chained = chain_groups(c, cfg, O, P.maxcoord);
    const Chains chains = chain_table(c, cfg, in, P, O, chained, ev_matches, exact_host, S);
    const KeptChains kc = order_chains(c, cfg, in, P, chains, exact_host, S);

    stage_mark(c, "assign+inversion+rescue");
    // The anchor pass hands the inversion capture its candidates when it visits every alive record (every alive record is a
    // sorted position) and the capture walks the chains of a pair (not the buckets of inversion_grid, which sorts them itself).
    const bool capture = !cfg.scaffolds_only && kc.C2 > 0;
    const bool fused_candidates = capture && O.n_m == P.n_alive && !takes_inversion_grid(c, cfg, P, chained.n_huge);
    const InvCands cands = assign_anchors(c, O, chains, P.flags, status, chain_id, fused_candidates);
    if (capture) {
        capture_inversions(c, cfg, in, P, chained.n_huge, kc, cands, status, chain_id);
        if (cfg.scaffold_max_deviation > 0) rescue(c, cfg, in, P, status, chain_id);
    }

    // k_assign, the inversion capture and rescue have counted the statuses they wrote (C_ANCHORS, C_RESCUED)
    stage_mark(c, "stats");
    read_counters(c);
    S.n_anchors = c->h_ctr[C_ANCHORS];
    S.n_rescued = c->h_ctr[C_RESCUED];
    S.n_kept = S.n_anchors + S.n_rescued;
    S.score_near_ties = c->h_ctr[C_NEAR_TIES];
    finish(c, S, launches0, stats);
}

// ---- does the device's ln() produce the host libm's bits? ------------------------------------------
// 2^16 probe arguments: every integer up to 2^15 and pseudo-random integers up to 2^32 (spans and gaps are integers).
struct t_probe;
static bool probe_log(swg_ctx *c) {
    const u32 n = 1u << 16;
    c->arena.reserve((size_t)n * 32 + (1u << 20));
    double *d = c->arena.take<double>(2 * (size_t)n);
    launch_for<t_probe>(n, c->stream, c->lc, [=] __device__(u32 k) {
        u64 x = k < (1u << 15) ? (u64)k + 1 : ((u64)k * 0x9E3779B97F4A7C15ull >> 32) + 2;
        d[k] = ln_fn((double)x, false);
        d[n + k] = ln_fn((double)x, true);
    });
    std::vector<double> h(2 * (size_t)n);
    SWG_CUDA(cudaMemcpyAsync(h.data(), d, sizeof(double) * 2 * n, cudaMemcpyDeviceToHost, c->stream));
    SWG_CUDA(cudaStreamSynchronize(c->stream));
    bool port_ok = true, cuda_ok = true;
    for (u32 k = 0; k < n; k++) {
        const u64 x = k < (1u << 15) ? (u64)k + 1 : ((u64)k * 0x9E3779B97F4A7C15ull >> 32) + 2;
        const double ref = std::log((double)x);
        port_ok &= std::memcmp(&ref, &h[k], 8) == 0;
        cuda_ok &= std::memcmp(&ref, &h[n + k], 8) == 0;
    }
    c->cudalog_matches_host = cuda_ok;
    return port_ok;
}

// ---- the filter with the exact re-rank around it (DESIGN 4d) ---------------------------------------
// Normal case: one run_filter.  If a sweep saw two scores within NEAR_TIE_ULPS of each other AND the device's ln() is not
// known to equal the host libm's (another glibc, SWG_LOG_IMPL=cuda), a ranking could differ from the reference's by one
// rounding: the call is redone with every logarithm computed by the HOST libm — the record scores as a column
// (identity * ln(span), all host threads), the chain-level ones inside run_filter.  SWG_EXACT_SCORES=always / never.
// host_*: the caller's host columns when it has them (swg_filter), else NULL (they are downloaded).
static void run_filter_exact(swg_ctx *c, const swg_config &cfg, const DevIn &in, u8 *status, u32 *chain_id, swg_stats *stats, cudaEvent_t ev_matches,
                             const swg_mappings *host) {
    const Knobs &K = c->knobs;
    const bool log_ok = K.cuda_log ? c->cudalog_matches_host : c->log_matches_host;
    const bool can = !in.score && in.n > 0;
    swg_stats first;
    std::memset(&first, 0, sizeof first);
    if (!(can && K.exact_scores == 1)) {
        run_filter(c, cfg, in, status, chain_id, &first, ev_matches);
        if (stats) *stats = first;
        if (!can || K.exact_scores == 2 || first.score_near_ties == 0 || log_ok) return;
    }
    const u32 n = in.n;
    if (ev_matches) SWG_CUDA(cudaStreamWaitEvent(c->stream, ev_matches, 0));
    std::vector<u32> hqs, hqe, hbl, hmt;
    std::vector<double> hid;
    const u32 *qs = host ? host->query_start : nullptr, *qe = host ? host->query_end : nullptr;
    const u32 *bl = host ? host->block_length : nullptr, *mt = host ? host->matches : nullptr;
    const double *id = host ? host->identity : nullptr;
    if (!host) {
        auto down = [&](auto &vec, const void *src, size_t bytes) { vec.resize(n); SWG_CUDA(cudaMemcpyAsync(vec.data(), src, bytes, cudaMemcpyDeviceToHost, c->stream)); };
        down(hqs, in.qs, (size_t)n * 4); down(hqe, in.qe, (size_t)n * 4);
        if (in.identity) down(hid, in.identity, (size_t)n * 8);
        else { down(hbl, in.blen, (size_t)n * 4); down(hmt, in.matches, (size_t)n * 4); }
        SWG_CUDA(cudaStreamSynchronize(c->stream));
        qs = hqs.data(); qe = hqe.data();
        id = in.identity ? hid.data() : nullptr;
        bl = hbl.data(); mt = hmt.data();
    }
    c->h_score.resize(n);
    {
        const int scoring = cfg.scoring_function;
        const unsigned nt = std::max(1u, std::min(16u, std::thread::hardware_concurrency()));
        std::vector<std::thread> th;
        double *out = c->h_score.data();
        for (unsigned t = 0; t < nt; t++)
            th.emplace_back([=]() {
                const size_t a = (size_t)n * t / nt, b = (size_t)n * (t + 1) / nt;
                for (size_t i = a; i < b; i++) {
                    const double idv = id ? id[i] : (double)mt[i] / (double)(bl[i] > 1 ? bl[i] : 1);
                    out[i] = host_score(scoring, idv, qs[i], qe[i]);
                }
            });
        for (auto &t : th) t.join();
    }
    c->score_arena.reserve((size_t)n * 8 + 1024);
    double *d_score = c->score_arena.take<double>(n);
    SWG_CUDA(cudaMemcpyAsync(d_score, c->h_score.data(), (size_t)n * 8, cudaMemcpyHostToDevice, c->stream));
    DevIn in2 = in;
    in2.score = d_score;
    swg_stats second;
    run_filter(c, cfg, in2, status, chain_id, &second, nullptr, true);
    second.exact_rerank = 1;
    second.gpu_launches += first.gpu_launches;
    if (stats) *stats = second;
}

static int guarded(swg_ctx *c, const char *what, void (*fn)(void *), void *arg) {
    struct DrainCopies { // an error must not leave the caller's host buffers in use by an in-flight copy
        swg_ctx *c;
        ~DrainCopies() { if (c && c->copy_stream) cudaStreamSynchronize(c->copy_stream); }
    } drain{c};
    try {
        if (c) c->knobs = read_knobs();
        fn(arg);
        return SWG_OK;
    } catch (const CudaError &e) {
        set_err(c, std::string(what) + ": CUDA error '" + cudaGetErrorString(e.code) + "' at " + e.file + ":" + std::to_string(e.line));
        cudaGetLastError();
        return SWG_ERR_CUDA;
    } catch (const RangeError &e) {
        set_err(c, std::string(what) + ": " + e.msg);
        return SWG_ERR_RANGE;
    } catch (const IoError &e) {
        set_err(c, std::string(what) + ": " + e.msg);
        return SWG_ERR_IO;
    } catch (const OomError &e) {
        set_err(c, std::string(what) + ": out of device memory (" + std::to_string(e.bytes) + " bytes)");
        return SWG_ERR_OOM;
    } catch (const std::bad_alloc &) {
        set_err(c, std::string(what) + ": out of host memory");
        return SWG_ERR_OOM;
    }
}

static bool check_cfg(swg_ctx *c, const swg_config *cfg) {
    if (!cfg || cfg->mapping_filter_mode > 2 || cfg->scaffold_filter_mode > 2 || cfg->scoring_function > 4) {
        set_err(c, "bad swg_config (NULL or enum out of range)");
        return false;
    }
    return true;
}
static bool check_maps(swg_ctx *c, const swg_mappings *m) {
    if (!m) { set_err(c, "NULL swg_mappings"); return false; }
    if (m->n == 0) return true;
    if (m->n >= 0x7FFFFFF0ull) { set_err(c, "n too large (must be < 2^31 per context)"); return false; }
    const bool ids32 = m->query_id && m->target_id, ids16 = !m->query_id && !m->target_id && m->query_id16 && m->target_id16 && m->n_seq <= 65536;
    if (!(ids32 || ids16) || !m->query_start || !m->query_end || !m->target_start || !m->target_end ||
        !m->block_length || !m->matches || !m->strand || !m->seq_genome_id || !m->seq_genome2_id || m->n_seq == 0) { // identity may be NULL
        set_err(c, "swg_mappings has a NULL column or n_seq == 0");
        return false;
    }
    return true;
}
static DevIn make_devin(const swg_mappings *m) {
    DevIn d;
    d.qid = m->query_id; d.tid = m->target_id; d.qs = m->query_start; d.qe = m->query_end; d.ts = m->target_start;
    d.te = m->target_end; d.blen = m->block_length; d.matches = m->matches; d.identity = m->identity; d.strand = m->strand;
    d.score = m->score; d.P = m->seq_genome_id; d.P2 = m->seq_genome2_id; d.n = (u32)m->n; d.n_seq = m->n_seq;
    return d;
}

// ---- host <-> device copies through pinned pieces (pageable caller memory, file text) --------------------------------------
// cudaMemcpyAsync from PAGEABLE memory is staged by the driver on one thread (a few GB/s, and it blocks); a Rust Vec or a numpy
// array is pageable.  Here a team of threads copies 8 MiB pieces into pinned buffers and queues one DMA per piece, so the link
// stays busy: the path swg_filter takes whenever a caller's column is not page-locked.
static constexpr size_t PIN_PIECE = (size_t)8 << 20;
static constexpr int PIN_COUNT = 12;

static void ensure_pinned(swg_ctx *c) {
    if (!c->pin.empty()) return;
    for (int i = 0; i < PIN_COUNT; i++) {
        char *p = nullptr;
        SWG_CUDA(cudaMallocHost(&p, PIN_PIECE));
        c->pin.push_back(p);
        cudaEvent_t e;
        SWG_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        c->pin_ev.push_back(e);
    }
}
struct CopyJob { const char *src; char *dst; size_t bytes; int fd; }; // fd >= 0: the source is that file (pread), src its mapping

// The general form: one column is one contiguous device range whose bytes come from (or go to) several host slices, e.g. the
// same column of many tables (swg_filter_batch).  seg.off is the slice's byte offset inside the column; slices are ascending
// and disjoint.  A piece is PIN_PIECE bytes of ONE column and one DMA, however many slices it covers.
struct PinSeg { char *host; size_t off, len; int fd = -1; }; // fd >= 0: host -> device reads the slice from that file (pread)
struct PinCol { char *dev; size_t bytes; std::vector<PinSeg> segs; };
struct PinPiece { const PinCol *col; size_t off, len, seg0; };
static std::vector<PinPiece> pin_pieces(const std::vector<PinCol> &cols) {
    std::vector<PinPiece> pieces;
    for (const PinCol &col : cols) {
        size_t s = 0;
        for (size_t o = 0; o < col.bytes; o += PIN_PIECE) {
            while (s < col.segs.size() && col.segs[s].off + col.segs[s].len <= o) s++;
            pieces.push_back(PinPiece{&col, o, std::min(PIN_PIECE, col.bytes - o), s});
        }
    }
    return pieces;
}
// fn(slice, byte offset inside the slice, byte offset inside the piece, length) for every slice the piece overlaps
template <class F> static void piece_slices(const PinPiece &p, F fn) {
    const std::vector<PinSeg> &segs = p.col->segs;
    for (size_t s = p.seg0; s < segs.size() && segs[s].off < p.off + p.len; s++) {
        const size_t a = std::max(segs[s].off, p.off), b = std::min(segs[s].off + segs[s].len, p.off + p.len);
        if (a < b) fn(segs[s], a - segs[s].off, a - p.off, b - a);
    }
}
static std::vector<PinCol> jobs_as_cols(const std::vector<CopyJob> &jobs, bool h2d) {
    std::vector<PinCol> cols;
    for (const CopyJob &j : jobs)
        cols.push_back(h2d ? PinCol{j.dst, j.bytes, {PinSeg{(char *)j.src, 0, j.bytes, j.fd}}} : PinCol{(char *)j.src, j.bytes, {PinSeg{j.dst, 0, j.bytes, -1}}});
    return cols;
}

// host -> device on c->copy_stream; returns when every piece is QUEUED (the last DMAs may still be in flight).  Bytes of a piece
// that no slice covers carry whatever the pinned buffer held.
static void staged_h2d_cols(swg_ctx *c, const std::vector<PinCol> &cols) {
    ensure_pinned(c);
    const std::vector<PinPiece> pieces = pin_pieces(cols);
    std::atomic<size_t> next{0};
    std::atomic<int> failed{0};
    auto worker = [&](int t) {
        cudaSetDevice(c->device);
        while (!failed.load()) {
            const size_t k = next.fetch_add(1);
            if (k >= pieces.size()) break;
            const PinPiece &pc = pieces[k];
            if (cudaEventSynchronize(c->pin_ev[t]) != cudaSuccess) { failed = 1; break; }
            char *buf = c->pin[t];
            piece_slices(pc, [&](const PinSeg &sg, size_t so, size_t po, size_t len) {
                bool filled = false;
                if (sg.fd >= 0) { // plain file: pread skips the page-table work of touching a fresh mapping
                    size_t got = 0;
                    while (got < len) {
                        const ssize_t r = pread(sg.fd, buf + po + got, len - got, (off_t)(so + got));
                        if (r <= 0) break;
                        got += (size_t)r;
                    }
                    filled = got == len;
                }
                if (!filled) memcpy(buf + po, sg.host + so, len);
            });
            if (cudaMemcpyAsync(pc.col->dev + pc.off, buf, pc.len, cudaMemcpyHostToDevice, c->copy_stream) != cudaSuccess ||
                cudaEventRecord(c->pin_ev[t], c->copy_stream) != cudaSuccess) { failed = 1; break; }
        }
    };
    std::vector<std::thread> th;
    const int nt = (int)std::min<size_t>(PIN_COUNT, pieces.size());
    for (int t = 1; t < nt; t++) th.emplace_back(worker, t);
    if (nt > 0) worker(0);
    for (auto &t : th) t.join();
    if (failed.load()) { cudaGetLastError(); throw CudaError{cudaErrorUnknown, __FILE__, __LINE__}; }
}
static void staged_h2d(swg_ctx *c, const std::vector<CopyJob> &jobs) { staged_h2d_cols(c, jobs_as_cols(jobs, true)); }
// device -> pageable host memory: DMA per piece into a pinned buffer, the team copies the slices out; returns when done.
// The device data must be complete on c->copy_stream's view (the caller makes copy_stream wait for the producing stream).
static void staged_d2h_cols(swg_ctx *c, const std::vector<PinCol> &cols) {
    ensure_pinned(c);
    const std::vector<PinPiece> pieces = pin_pieces(cols);
    std::atomic<size_t> next{0};
    std::atomic<int> failed{0};
    auto worker = [&](int t) {
        cudaSetDevice(c->device);
        while (!failed.load()) {
            const size_t k = next.fetch_add(1);
            if (k >= pieces.size()) break;
            const PinPiece &pc = pieces[k];
            char *buf = c->pin[t];
            if (cudaMemcpyAsync(buf, pc.col->dev + pc.off, pc.len, cudaMemcpyDeviceToHost, c->copy_stream) != cudaSuccess ||
                cudaEventRecord(c->pin_ev[t], c->copy_stream) != cudaSuccess || cudaEventSynchronize(c->pin_ev[t]) != cudaSuccess) { failed = 1; break; }
            piece_slices(pc, [&](const PinSeg &sg, size_t so, size_t po, size_t len) { memcpy(sg.host + so, buf + po, len); });
        }
    };
    std::vector<std::thread> th;
    const int nt = (int)std::min<size_t>(PIN_COUNT, pieces.size());
    for (int t = 1; t < nt; t++) th.emplace_back(worker, t);
    if (nt > 0) worker(0);
    for (auto &t : th) t.join();
    if (failed.load()) { cudaGetLastError(); throw CudaError{cudaErrorUnknown, __FILE__, __LINE__}; }
}
static void staged_d2h(swg_ctx *c, const std::vector<CopyJob> &jobs /* src = device, dst = host */) { staged_d2h_cols(c, jobs_as_cols(jobs, false)); }
static bool is_pageable(const void *p) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return true; }
    return at.type == cudaMemoryTypeUnregistered;
}

struct UploadArgs { swg_ctx *c; const swg_mappings *in; swg_mappings *dev; swg_result *res; Arena *arena; bool overlap_matches = false; size_t h2d_bytes = 0; bool pageable = false;
                    cudaStream_t stream = nullptr; /* NULL: the context's main stream */
                    bool late_blen = false; /* block_length travels with `matches` (the retain does not test it: min_block_length == 0) */ };

struct t_widen;
static void do_upload(void *p) {
    UploadArgs *a = (UploadArgs *)p;
    swg_ctx *c = a->c;
    const swg_mappings *h = a->in;
    SWG_CUDA(cudaSetDevice(c->device));
    size_t n = h->n;
    const bool id16 = h->query_id == nullptr; // 16-bit id columns (n_seq <= 65536): 2 B instead of 4 B per id on the wire
    const size_t idb = id16 ? 2 : 4;
    size_t bytes = n * (8 * 4 + (id16 ? 4 + 8 : 0) + (h->identity ? 8 : 0) + 1 + (h->score ? 8 : 0) + 1 + 4) + (size_t)h->n_seq * 8 + 64 * 256;
    a->h2d_bytes = n * (6 * 4 + 2 * idb + (h->identity ? 8 : 0) + 1 + (h->score ? 8 : 0)) + (size_t)h->n_seq * 8;
    a->arena->reserve(bytes);
    Arena &A = *a->arena;
    swg_mappings d = *h;
    cudaStream_t st = a->stream ? a->stream : c->stream;
    // the columns the first kernels need, then `matches` (first read after the sort): with overlap_matches it travels behind the
    // others on the copy stream, so prefilter, key build and sort run while it is still on the wire
    std::vector<CopyJob> first, last;
    auto col = [&](const void *src, size_t cnt, size_t elem, std::vector<CopyJob> &jobs) {
        char *dst = A.take<char>(cnt * elem);
        jobs.push_back(CopyJob{(const char *)src, dst, cnt * elem, -1});
        return (void *)dst;
    };
    u16 *q16 = nullptr, *t16 = nullptr;
    if (id16) { q16 = (u16 *)col(h->query_id16, n, 2, first); t16 = (u16 *)col(h->target_id16, n, 2, first); }
    else { d.query_id = (const u32 *)col(h->query_id, n, 4, first); d.target_id = (const u32 *)col(h->target_id, n, 4, first); }
    d.query_start = (const u32 *)col(h->query_start, n, 4, first); d.query_end = (const u32 *)col(h->query_end, n, 4, first);
    d.target_start = (const u32 *)col(h->target_start, n, 4, first); d.target_end = (const u32 *)col(h->target_end, n, 4, first);
    if (!(a->overlap_matches && a->late_blen)) d.block_length = (const u32 *)col(h->block_length, n, 4, first);
    if (h->identity) d.identity = (const double *)col(h->identity, n, 8, first);
    if (h->score) d.score = (const double *)col(h->score, n, 8, first);
    d.strand = (const u8 *)col(h->strand, n, 1, first);
    d.seq_genome_id = (const u32 *)col(h->seq_genome_id, h->n_seq, 4, first);
    d.seq_genome2_id = (const u32 *)col(h->seq_genome2_id, h->n_seq, 4, first);
    a->res->status = A.take<u8>(n);
    a->res->chain_id = A.take<u32>(n);
    d.matches = (const u32 *)col(h->matches, n, 4, last);
    if (a->overlap_matches && a->late_blen) d.block_length = (const u32 *)col(h->block_length, n, 4, last);
    bool pageable = false;
    for (const CopyJob &j : first) pageable |= j.bytes >= (1u << 20) && is_pageable(j.src);
    for (const CopyJob &j : last) pageable |= j.bytes >= (1u << 20) && is_pageable(j.src);
    if (pageable) {
        // pinned pieces on the copy stream (behind whatever the main stream has queued), the main stream waits for them
        SWG_CUDA(cudaEventRecord(c->ev_copy[0], st));
        SWG_CUDA(cudaStreamWaitEvent(c->copy_stream, c->ev_copy[0], 0));
        staged_h2d(c, first);
        SWG_CUDA(cudaEventRecord(c->ev_copy[0], c->copy_stream));
        SWG_CUDA(cudaStreamWaitEvent(st, c->ev_copy[0], 0));
        staged_h2d(c, last);
        SWG_CUDA(cudaEventRecord(c->ev_copy[1], c->copy_stream));
        if (!a->overlap_matches) SWG_CUDA(cudaStreamWaitEvent(st, c->ev_copy[1], 0));
    } else {
        for (const CopyJob &j : first) SWG_CUDA(cudaMemcpyAsync(j.dst, j.src, j.bytes, cudaMemcpyHostToDevice, st));
        cudaStream_t cs = st;
        if (a->overlap_matches) {
            SWG_CUDA(cudaEventRecord(c->ev_copy[0], st));
            SWG_CUDA(cudaStreamWaitEvent(c->copy_stream, c->ev_copy[0], 0));
            cs = c->copy_stream;
        }
        for (const CopyJob &j : last) SWG_CUDA(cudaMemcpyAsync(j.dst, j.src, j.bytes, cudaMemcpyHostToDevice, cs));
        if (a->overlap_matches) SWG_CUDA(cudaEventRecord(c->ev_copy[1], cs));
    }
    if (id16) { // widen on the device: every kernel reads 32-bit ids
        u32 *q32 = A.take<u32>(n), *t32 = A.take<u32>(n);
        launch_for<t_widen>((u32)n, st, c->lc, [=] __device__(u32 i) { q32[i] = q16[i]; t32[i] = t16[i]; });
        d.query_id = q32;
        d.target_id = t32;
    }
    a->pageable = pageable;
    *a->dev = d;
}


struct SweepArgs {
    swg_ctx *c; uint64_t n; const uint32_t *qs, *qe, *ts, *te; const double *identity;
    uint64_t nq, nt; double thr; int scoring; int axis; uint8_t *keep;
};
static void do_sweep(void *p) {
    SweepArgs *a = (SweepArgs *)p;
    swg_ctx *c = a->c;
    SWG_CUDA(cudaSetDevice(c->device));
    u32 n = (u32)a->n;
    if (n == 0) return;
    cudaStream_t st = c->stream;
    c->arena.reserve((size_t)n * 200 + (16u << 20));
    Arena &A = c->arena;
    u32 *qs = A.take<u32>(n), *qe = A.take<u32>(n), *ts = A.take<u32>(n), *te = A.take<u32>(n);
    double *id = A.take<double>(n), *score = A.take<double>(n);
    u64 *gk = A.take<u64>(n);
    u8 *k1 = A.take<u8>(n), *k2 = A.take<u8>(n);
    SWG_CUDA(cudaMemcpyAsync(qs, a->qs, n * 4, cudaMemcpyHostToDevice, st));
    SWG_CUDA(cudaMemcpyAsync(qe, a->qe, n * 4, cudaMemcpyHostToDevice, st));
    SWG_CUDA(cudaMemcpyAsync(ts, a->ts, n * 4, cudaMemcpyHostToDevice, st));
    SWG_CUDA(cudaMemcpyAsync(te, a->te, n * 4, cudaMemcpyHostToDevice, st));
    SWG_CUDA(cudaMemcpyAsync(id, a->identity, n * 8, cudaMemcpyHostToDevice, st));
    SWG_CUDA(cudaMemsetAsync(gk, 0, sizeof(u64) * n, st));
    SWG_CUDA(cudaMemsetAsync(c->d_ctr, 0, sizeof(u64) * C_COUNT, st));
    const int scoring = a->scoring;
    launch_for<t_scores>(n, st, c->lc, [=] __device__(u32 i) { score[i] = score_fn(scoring, id[i], qs[i], qe[i]); });
    u8 *res = k1;
    if (a->axis == 0) general_sweep(c, n, nullptr, 0, gk, 1, 32, qs, qe, score, a->nq, a->thr, k1);
    else if (a->axis == 1) general_sweep(c, n, nullptr, 0, gk, 1, 32, ts, te, score, a->nt, a->thr, k1);
    else {
        general_sweep(c, n, nullptr, 0, gk, 1, 32, qs, qe, score, a->nq, a->thr, k1);
        general_sweep(c, n, k1, 1, gk, 1, 32, ts, te, score, a->nt, a->thr, k2);
        res = k2;
    }
    SWG_CUDA(cudaMemcpyAsync(a->keep, res, n, cudaMemcpyDeviceToHost, st));
    SWG_CUDA(cudaStreamSynchronize(st));
}

struct CoreArgs { swg_ctx *c; u64 n; const u32 *b, *e; const double *s; u64 max_keep; double thr; u64 *out; u64 *n_out; };
static void do_sweep_core(void *p) {
    CoreArgs *a = (CoreArgs *)p;
    swg_ctx *c = a->c;
    const u32 n = (u32)a->n;
    *a->n_out = 0;
    if (n == 0) return;
    if (n == 1) { a->out[0] = 0; *a->n_out = 1; return; }                       // plane_sweep_core.rs:89-91
    if (a->max_keep == SWG_KEEP_ALL) { for (u32 i = 0; i < n; i++) a->out[i] = i; *a->n_out = n; return; } // :94-96
    SWG_CUDA(cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    c->arena.reserve((size_t)n * 160 + (16u << 20));
    Arena &A = c->arena;
    u32 *b = A.take<u32>(n), *e = A.take<u32>(n);
    double *sc = A.take<double>(n);
    SWG_CUDA(cudaMemcpyAsync(b, a->b, n * 4, cudaMemcpyHostToDevice, st));
    SWG_CUDA(cudaMemcpyAsync(e, a->e, n * 4, cudaMemcpyHostToDevice, st));
    SWG_CUDA(cudaMemcpyAsync(sc, a->s, n * 8, cudaMemcpyHostToDevice, st));
    u64 *ek = A.take<u64>(2 * n), *ek2 = A.take<u64>(2 * n);
    u32 *ev = A.take<u32>(2 * n), *ev2 = A.take<u32>(2 * n);
    launch_for<t_events>(n, st, c->lc, [=] __device__(u32 i) {
        ek[2 * i] = (u64)b[i] << 1; ev[2 * i] = 2 * i;
        ek[2 * i + 1] = ((u64)e[i] << 1) | 1; ev[2 * i + 1] = 2 * i + 1;
    });
    sort_pairs(c, ek, ek2, ev, ev2, 2 * n, 33); // stable: equal (pos,type) keep index order
    CoreEntry *act = A.take<CoreEntry>(n + 1);
    u8 *marked = A.take<u8>(n);
    SWG_CUDA(cudaMemsetAsync(marked, 0, n, st));
    k_sweep_core_mark<<<1, 32, 0, st>>>(ev, 2 * n, sc, a->max_keep, act, marked);
    c->lc.n++;
    // marked set in ascending index order
    u32 *list = A.take<u32>(n), *bsum = A.take<u32>(scan_temp_u32(n)), *d_cnt = A.take<u32>(2);
    scan_flags([=] __device__(u32 i) -> u32 { return marked[i] ? 1u : 0u; }, [=] __device__(u32 i, u32 ex, u32 v) { if (v) list[ex] = i; },
               n, bsum, d_cnt, st, c->lc);
    u32 nk = read_u32(c, d_cnt);
    std::vector<u32> host(nk);
    if (a->thr < 1.0 && nk > 1) {
        u64 *sk = A.take<u64>(nk), *sk2 = A.take<u64>(nk);
        u32 *sv = A.take<u32>(nk), *sv2 = A.take<u32>(nk);
        launch_for<t_iota>(nk, st, c->lc, [=] __device__(u32 t) { sk[t] = score_desc_key(sc[list[t]]); sv[t] = list[t]; });
        sort_pairs(c, sk, sk2, sv, sv2, nk, 64);
        u32 *acc = A.take<u32>(nk);
        k_sweep_core_greedy<<<1, 32, 0, st>>>(sv, nk, b, e, a->thr, acc, d_cnt + 1);
        c->lc.n++;
        nk = read_u32(c, d_cnt + 1);
        host.resize(nk);
        SWG_CUDA(cudaMemcpyAsync(host.data(), acc, nk * 4, cudaMemcpyDeviceToHost, st));
    } else if (nk) {
        SWG_CUDA(cudaMemcpyAsync(host.data(), list, nk * 4, cudaMemcpyDeviceToHost, st));
    }
    SWG_CUDA(cudaStreamSynchronize(st));
    for (u32 i = 0; i < nk; i++) a->out[i] = host[i];
    *a->n_out = nk;
}

} // namespace swg

#include "paf_device.cuh"
#include "ani_device.cuh"
#include "batch.cuh"

namespace swg {

// Opens the text of a PAF input for the entry point `who`.  On failure the error is set and the code returned:
// SWG_ERR_RANGE when the file is readable (so its contents are at fault), SWG_ERR_IO otherwise.
static int open_paf_text(swg_ctx *c, const char *who, const char *path, swg_paf *hp) {
    std::string err;
    if (paf_open_text(path, hp, &err)) return SWG_OK;
    set_err(c, std::string(who) + ": " + err);
    return access(path, R_OK) == 0 ? SWG_ERR_RANGE : SWG_ERR_IO;
}

// The device readers without a host front end (swg_ani_stats, swg_tree_filter_paf): run() catches their declines, rc()
// turns them into the return code.
struct Declines {
    bool fallback = false, nan = false;
    template <class F> void run(F &&f) {
        try { f(); } catch (const FrontEndFallback &) { fallback = true; } catch (const NanError &) { nan = true; }
    }
    int rc(swg_ctx *c, const char *who, const char *nan_what) const {
        if (nan) { set_err(c, std::string(who) + ": " + nan_what + " (the reference panics here)"); return SWG_ERR_RANGE; }
        if (fallback) {
            set_err(c, std::string(who) + ": input not supported by the device front end (> 64 GiB, or a sequence-name hash collision)");
            return SWG_ERR_UNSUPPORTED;
        }
        return SWG_OK;
    }
};

} // namespace swg

// =================================================================================================
// C ABI
// =================================================================================================
extern "C" {

swg_ctx *swg_create(int device) {
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        g_create_error = std::string("swg_create: no usable CUDA device (") + cudaGetErrorString(e) + "); this library has no CPU fallback";
        cudaGetLastError();
        return nullptr;
    }
    if (device < 0 || device >= ndev) { g_create_error = "swg_create: device index out of range"; return nullptr; }
    swg_ctx *c = new (std::nothrow) swg_ctx();
    if (!c) return nullptr;
    c->device = device;
    try {
        SWG_CUDA(cudaSetDevice(device));
        cudaDeviceProp prop;
        SWG_CUDA(cudaGetDeviceProperties(&prop, device));
        if (prop.major < 10) throw RangeError{"device is not sm_100 class (this build carries sm_100a code only)"};
        c->sm_count = prop.multiProcessorCount;
        SWG_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
        for (auto &ev : c->ev) SWG_CUDA(cudaEventCreate(&ev));
        for (auto &ev : c->ev_sort) SWG_CUDA(cudaEventCreate(&ev));
        for (auto &ev : c->ev_pre) SWG_CUDA(cudaEventCreate(&ev));
        SWG_CUDA(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
        SWG_CUDA(cudaStreamCreateWithFlags(&c->up_stream, cudaStreamNonBlocking));
        for (auto &p : c->pf) SWG_CUDA(cudaEventCreateWithFlags(&p.ready, cudaEventDisableTiming));
        for (auto &ev : c->ev_copy) SWG_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        SWG_CUDA(cudaEventCreateWithFlags(&c->ev_ctr, cudaEventDisableTiming));
        SWG_CUDA(cudaMallocHost(&c->h_ctr, sizeof(u64) * (C_COUNT + 8)));
        SWG_CUDA(cudaMalloc(&c->d_ctr, sizeof(u64) * C_COUNT));
        rs_init_device(); // dynamic shared memory opt-in of the one-sweep kernels: a per-device attribute
        gs_init_device();
        c->knobs = read_knobs();
        c->log_matches_host = probe_log(c);
    } catch (const CudaError &e2) {
        g_create_error = std::string("swg_create: CUDA error '") + cudaGetErrorString(e2.code) + "'";
        delete c;
        return nullptr;
    } catch (const RangeError &e3) {
        g_create_error = "swg_create: " + e3.msg;
        delete c;
        return nullptr;
    }
    return c;
}

void swg_destroy(swg_ctx *c) {
    if (!c) return;
    cudaSetDevice(c->device);
    c->arena.release();
    c->io.release();
    c->keys.release();
    c->batch.release();
    c->score_arena.release();
    if (c->h_ctr) cudaFreeHost(c->h_ctr);
    for (char *p : c->pin) cudaFreeHost(p);
    for (auto &ev : c->pin_ev) cudaEventDestroy(ev);
    if (c->d_ctr) cudaFree(c->d_ctr);
    if (c->gtable) cudaFree(c->gtable);
    for (auto &ev : c->ev) if (ev) cudaEventDestroy(ev);
    for (auto &ev : c->ev_sort) if (ev) cudaEventDestroy(ev);
    for (auto &ev : c->ev_pre) if (ev) cudaEventDestroy(ev);
    for (auto &ev : c->ev_copy) if (ev) cudaEventDestroy(ev);
    if (c->ev_ctr) cudaEventDestroy(c->ev_ctr);
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    if (c->up_stream) { cudaStreamSynchronize(c->up_stream); cudaStreamDestroy(c->up_stream); }
    for (auto &p : c->pf) { if (p.ready) cudaEventDestroy(p.ready); p.arena.release(); }
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
}

void swg__set_error(swg_ctx *c, const char *msg) { set_err(c, msg ? msg : ""); }
const char *swg_last_error(const swg_ctx *c) { return c ? c->err.c_str() : g_create_error.c_str(); }
void *swg_stream(swg_ctx *c) { return c ? (void *)c->stream : nullptr; }

struct FilterDevArgs { swg_ctx *c; const swg_config *cfg; const swg_mappings *in; swg_result *out; swg_stats *stats; };

int swg_filter_device(swg_ctx *c, const swg_config *cfg, const swg_mappings *dev_in, swg_result *dev_out, swg_stats *stats) {
    if (!c) return SWG_ERR_ARG;
    if (!check_cfg(c, cfg) || !check_maps(c, dev_in) || !dev_out || (dev_in->n && (!dev_out->status || !dev_out->chain_id))) return SWG_ERR_ARG;
    FilterDevArgs a{c, cfg, dev_in, dev_out, stats};
    return guarded(c, "swg_filter_device", [](void *p) {
        FilterDevArgs *a = (FilterDevArgs *)p;
        SWG_CUDA(cudaSetDevice(a->c->device));
        SWG_CUDA(cudaEventRecord(a->c->ev[1], a->c->stream));
        swg_stats local;
        run_filter_exact(a->c, *a->cfg, make_devin(a->in), a->out->status, a->out->chain_id, &local, nullptr, nullptr);
        if (a->stats) *a->stats = local;
        SWG_CUDA(cudaEventRecord(a->c->ev[2], a->c->stream));
        SWG_CUDA(cudaStreamSynchronize(a->c->stream));
        if (a->stats) {
            float ms = 0;
            SWG_CUDA(cudaEventElapsedTime(&ms, a->c->ev[1], a->c->ev[2]));
            a->stats->ms_device = ms;
        }
    }, &a);
}

int swg_filter(swg_ctx *c, const swg_config *cfg, const swg_mappings *host_in, swg_result *host_out, swg_stats *stats) {
    if (!c) return SWG_ERR_ARG;
    if (!check_cfg(c, cfg) || !check_maps(c, host_in) || !host_out || (host_in->n && (!host_out->status || !host_out->chain_id))) return SWG_ERR_ARG;
    struct Args { swg_ctx *c; const swg_config *cfg; const swg_mappings *in; swg_result *out; swg_stats *stats; } a{c, cfg, host_in, host_out, stats};
    return guarded(c, "swg_filter", [](void *p) {
        Args *a = (Args *)p;
        swg_ctx *c = a->c;
        SWG_CUDA(cudaSetDevice(c->device));
        swg_mappings dev;
        swg_result dres;
        UploadArgs ua{c, a->in, &dev, &dres, &c->io, true};
        ua.late_blen = a->cfg->min_block_length == 0;
        SWG_CUDA(cudaEventRecord(c->ev[0], c->stream));
        // a table swg_prefetch already put (or is putting) on the device: same n, same column pointers, oldest first
        swg_ctx::Prefetched *pf = nullptr;
        if (a->in->n && c->pf_count > 0) {
            swg_ctx::Prefetched &p = c->pf[c->pf_head];
            const swg_mappings &k = p.key, &m = *a->in;
            if (p.valid && k.n == m.n && k.n_seq == m.n_seq && k.query_id == m.query_id && k.target_id == m.target_id && k.query_id16 == m.query_id16 &&
                k.target_id16 == m.target_id16 && k.query_start == m.query_start && k.query_end == m.query_end && k.target_start == m.target_start &&
                k.target_end == m.target_end && k.block_length == m.block_length && k.matches == m.matches && k.identity == m.identity &&
                k.strand == m.strand && k.score == m.score && k.seq_genome_id == m.seq_genome_id && k.seq_genome2_id == m.seq_genome2_id)
                pf = &p;
        }
        if (pf) {
            dev = pf->dev;
            dres = pf->dres;
            ua.h2d_bytes = pf->h2d_bytes;
            SWG_CUDA(cudaStreamWaitEvent(c->stream, pf->ready, 0));
        } else if (a->in->n) do_upload(&ua);
        SWG_CUDA(cudaEventRecord(c->ev[1], c->stream));
        swg_stats local;
        std::memset(&local, 0, sizeof local);
        if (a->in->n) {
            run_filter_exact(c, *a->cfg, make_devin(&dev), dres.status, dres.chain_id, &local, pf ? nullptr : c->ev_copy[1], a->in);
            if (!pf) SWG_CUDA(cudaStreamWaitEvent(c->stream, c->ev_copy[1], 0)); // early exits never touched `matches`: still wait for its copy
        }
        SWG_CUDA(cudaEventRecord(c->ev[2], c->stream));
        if (a->in->n) {
            if (a->in->n * 5 >= (1u << 20) && (is_pageable(a->out->status) || is_pageable(a->out->chain_id))) {
                SWG_CUDA(cudaStreamWaitEvent(c->copy_stream, c->ev[2], 0));
                staged_d2h(c, std::vector<CopyJob>{CopyJob{(const char *)dres.status, (char *)a->out->status, (size_t)a->in->n, -1},
                                                    CopyJob{(const char *)dres.chain_id, (char *)a->out->chain_id, (size_t)a->in->n * 4, -1}});
                SWG_CUDA(cudaEventRecord(c->ev_copy[0], c->copy_stream));
                SWG_CUDA(cudaStreamWaitEvent(c->stream, c->ev_copy[0], 0));
            } else {
                SWG_CUDA(cudaMemcpyAsync(a->out->status, dres.status, a->in->n, cudaMemcpyDeviceToHost, c->stream));
                SWG_CUDA(cudaMemcpyAsync(a->out->chain_id, dres.chain_id, a->in->n * 4, cudaMemcpyDeviceToHost, c->stream));
            }
        }
        SWG_CUDA(cudaEventRecord(c->ev[3], c->stream));
        SWG_CUDA(cudaStreamSynchronize(c->stream));
        float m0 = 0, m1 = 0, m2 = 0;
        SWG_CUDA(cudaEventElapsedTime(&m0, c->ev[0], c->ev[1]));
        SWG_CUDA(cudaEventElapsedTime(&m1, c->ev[1], c->ev[2]));
        SWG_CUDA(cudaEventElapsedTime(&m2, c->ev[2], c->ev[3]));
        local.ms_h2d = m0; local.ms_device = m1; local.ms_d2h = m2;
        local.h2d_bytes = ua.h2d_bytes;
        local.d2h_bytes = a->in->n * 5;
        if (pf) { pf->valid = false; c->pf_head ^= 1; c->pf_count--; }
        if (a->stats) *a->stats = local;
    }, &a);
}

int swg_filter_batch(swg_ctx *c, const swg_config *cfg, uint64_t n_tables, const swg_mappings *host_in, swg_result *host_out,
                     uint64_t *table_counts, swg_stats *stats) {
    if (!c) return SWG_ERR_ARG;
    if (!check_cfg(c, cfg)) return SWG_ERR_ARG;
    if (n_tables && (!host_in || !host_out)) { set_err(c, "swg_filter_batch: NULL table or result array"); return SWG_ERR_ARG; }
    if (n_tables >= (1ull << 31)) { set_err(c, "swg_filter_batch: too many tables (must be < 2^31)"); return SWG_ERR_ARG; }
    u64 n = 0, n_seq = 0;
    int score = -1; // of the first non-empty table: every non-empty table has a score column, or none has
    for (u64 k = 0; k < n_tables; k++) {
        const swg_mappings &m = host_in[k];
        const std::string at = "swg_filter_batch: table " + std::to_string(k) + ": ";
        if (!check_maps(c, &m)) { set_err(c, at + c->err); return SWG_ERR_ARG; }
        if (m.n == 0) continue;
        if (!host_out[k].status || !host_out[k].chain_id) { set_err(c, at + "NULL result column"); return SWG_ERR_ARG; }
        if (score < 0) score = m.score != nullptr;
        if (score != (m.score != nullptr)) { set_err(c, at + "a score column must be given for every table or for none"); return SWG_ERR_ARG; }
        n += m.n;
        n_seq += m.n_seq;
        if (n >= 0x7FFFFFF0ull) { set_err(c, at + "the tables hold too many records together (must be < 2^31 per context)"); return SWG_ERR_ARG; }
        if (n_seq >= (1ull << 31)) { set_err(c, at + "the tables hold too many sequences together (must be < 2^31)"); return SWG_ERR_ARG; }
    }
    BatchArgs a{c, cfg, n_tables, host_in, host_out, table_counts, stats};
    return guarded(c, "swg_filter_batch", do_filter_batch, &a);
}

int swg_prefetch(swg_ctx *c, const swg_mappings *host_in) {
    if (!c) return SWG_ERR_ARG;
    if (!check_maps(c, host_in) || host_in->n == 0) return SWG_ERR_ARG;
    if (c->pf_count >= 2) { set_err(c, "swg_prefetch: two tables are already outstanding"); return SWG_ERR_ARG; }
    struct Args { swg_ctx *c; const swg_mappings *in; } a{c, host_in};
    return guarded(c, "swg_prefetch", [](void *p) {
        Args *a = (Args *)p;
        swg_ctx *c = a->c;
        SWG_CUDA(cudaSetDevice(c->device));
        swg_ctx::Prefetched &slot = c->pf[(c->pf_head + c->pf_count) & 1];
        UploadArgs ua{c, a->in, &slot.dev, &slot.dres, &slot.arena, false};
        ua.stream = c->up_stream;
        do_upload(&ua);
        SWG_CUDA(cudaEventRecord(slot.ready, c->up_stream));
        slot.key = *a->in;
        slot.h2d_bytes = ua.h2d_bytes;
        slot.valid = true;
        c->pf_count++;
    }, &a);
}
void swg_prefetch_drop(swg_ctx *c) {
    if (!c) return;
    cudaSetDevice(c->device);
    if (c->up_stream) cudaStreamSynchronize(c->up_stream);
    for (auto &p : c->pf) p.valid = false;
    c->pf_head = c->pf_count = 0;
}

int swg_upload(swg_ctx *c, const swg_mappings *host_in, swg_mappings *dev_out, swg_result *dev_res) {
    if (!c || !dev_out || !dev_res) return SWG_ERR_ARG;
    if (!check_maps(c, host_in) || host_in->n == 0) return SWG_ERR_ARG;
    Arena *ar = new (std::nothrow) Arena();
    if (!ar) return SWG_ERR_OOM;
    UploadArgs ua{c, host_in, dev_out, dev_res, ar};
    int rc = guarded(c, "swg_upload", [](void *p) { do_upload(p); SWG_CUDA(cudaStreamSynchronize(((UploadArgs *)p)->c->stream)); }, &ua);
    if (rc != SWG_OK) { ar->release(); delete ar; return rc; }
    // the arena base is the first column: recover it in swg_release from query_id
    delete ar; // (the device block itself stays allocated; base == dev_out->query_id)
    return SWG_OK;
}

void swg_release(swg_ctx *c, swg_mappings *dev, swg_result *dev_res) {
    if (!c || !dev) return;
    cudaSetDevice(c->device);
    if (dev->query_id) cudaFree((void *)dev->query_id);
    std::memset(dev, 0, sizeof *dev);
    if (dev_res) std::memset(dev_res, 0, sizeof *dev_res);
}

int swg_download_result(swg_ctx *c, uint64_t n, const swg_result *dev_res, swg_result *host_out) {
    if (!c || !dev_res || !host_out) return SWG_ERR_ARG;
    struct Args { swg_ctx *c; uint64_t n; const swg_result *d; swg_result *h; } a{c, n, dev_res, host_out};
    return guarded(c, "swg_download_result", [](void *p) {
        Args *a = (Args *)p;
        SWG_CUDA(cudaSetDevice(a->c->device));
        SWG_CUDA(cudaMemcpyAsync(a->h->status, a->d->status, a->n, cudaMemcpyDeviceToHost, a->c->stream));
        SWG_CUDA(cudaMemcpyAsync(a->h->chain_id, a->d->chain_id, a->n * 4, cudaMemcpyDeviceToHost, a->c->stream));
        SWG_CUDA(cudaStreamSynchronize(a->c->stream));
    }, &a);
}

int swg_last_chain_keys(swg_ctx *c, uint64_t cap, uint32_t *first_index_genome_pair, uint32_t *first_index_group, uint64_t *n_chains) {
    if (!c || !n_chains) return SWG_ERR_ARG;
    *n_chains = c->last_n_chains;
    if (c->last_n_chains == 0) return SWG_OK;
    if (cap < c->last_n_chains || !first_index_genome_pair || !first_index_group || !c->last_keyA) return SWG_ERR_ARG;
    struct Args { swg_ctx *c; uint32_t *a, *b; } a{c, first_index_genome_pair, first_index_group};
    return guarded(c, "swg_last_chain_keys", [](void *p) {
        Args *a = (Args *)p;
        SWG_CUDA(cudaSetDevice(a->c->device));
        SWG_CUDA(cudaMemcpyAsync(a->a, a->c->last_keyA, a->c->last_n_chains * 4, cudaMemcpyDeviceToHost, a->c->stream));
        SWG_CUDA(cudaMemcpyAsync(a->b, a->c->last_keyB, a->c->last_n_chains * 4, cudaMemcpyDeviceToHost, a->c->stream));
        SWG_CUDA(cudaStreamSynchronize(a->c->stream));
    }, &a);
}

// ---- multi-GPU merge helpers (SURVEY 8e: shards are unions of whole genome-pair units) -------------------------------
// The kept chains of one unit are numbered consecutively, on one GPU and in the merged numbering alike (order O3 sorts by the
// unit's first index A first), so merging needs only (A, count) per unit: swg_last_chain_units reports the runs of equal A
// among the kept chains of the last call (a few thousand values), swg_renumber_chains_device adds a per-run offset.
struct t_units; struct t_renumber; struct t_pack;
int swg_last_chain_units(swg_ctx *c, uint64_t cap, uint32_t *unit_first_index, uint32_t *unit_first_chain, uint64_t *n_units) {
    if (!c || !n_units) return SWG_ERR_ARG;
    struct Args { swg_ctx *c; u64 cap; u32 *a, *k; u64 *n; } a{c, cap, unit_first_index, unit_first_chain, n_units};
    return guarded(c, "swg_last_chain_units", [](void *p) {
        Args *a = (Args *)p;
        swg_ctx *c = a->c;
        *a->n = 0;
        const u32 C2 = (u32)c->last_n_chains;
        if (C2 == 0) return;
        SWG_CUDA(cudaSetDevice(c->device));
        // runs of equal A in chain order; the lists live behind the keys in the context-owned arena.  One round trip: the count
        // and the first min(cap, C2) entries of both lists travel together.
        u32 *run_k = c->keys.take<u32>(C2), *run_a = c->keys.take<u32>(C2), *bsum = c->keys.take<u32>(scan_temp_u32(C2)), *tot = c->keys.take<u32>(1);
        const u32 *kA = c->last_keyA;
        scan_flags([=] __device__(u32 u) -> bool { return u == 0 || kA[u] != kA[u - 1]; },
                   [=] __device__(u32 u, u32 ex, u32 v) { if (v) { run_k[ex] = u + 1; run_a[ex] = kA[u]; } }, C2, bsum, tot, c->stream, c->lc);
        u32 *h = reinterpret_cast<u32 *>(c->h_ctr + C_COUNT);
        SWG_CUDA(cudaMemcpyAsync(h, tot, sizeof(u32), cudaMemcpyDeviceToHost, c->stream));
        const u32 take = (u32)std::min<u64>(a->cap, C2);
        if (take && a->a && a->k) {
            SWG_CUDA(cudaMemcpyAsync(a->k, run_k, sizeof(u32) * take, cudaMemcpyDeviceToHost, c->stream)); // chain numbers are 1-based
            SWG_CUDA(cudaMemcpyAsync(a->a, run_a, sizeof(u32) * take, cudaMemcpyDeviceToHost, c->stream));
        }
        SWG_CUDA(cudaStreamSynchronize(c->stream));
        const u32 nu = *h;
        *a->n = nu;
        if (a->cap != 0 && (a->cap < nu || !a->a || !a->k)) throw RangeError{"capacity too small"};
    }, &a);
}
// chain_id[i] += delta[run of chain_id[i]] for every record with a chain (runs given by their first local chain number,
// ascending); chain_id is a DEVICE array of n entries, the two run arrays are HOST arrays.
int swg_renumber_chains_device(swg_ctx *c, uint64_t n, uint32_t *chain_id_dev, uint64_t n_units, const uint32_t *unit_first_chain,
                               const int64_t *unit_delta) {
    if (!c || (n && !chain_id_dev) || (n_units && (!unit_first_chain || !unit_delta)) || n >= 0x7FFFFFF0ull) return SWG_ERR_ARG;
    struct Args { swg_ctx *c; u32 n; u32 *ch; u32 nu; const u32 *fk; const int64_t *dl; } a{c, (u32)n, chain_id_dev, (u32)n_units, unit_first_chain, unit_delta};
    return guarded(c, "swg_renumber_chains_device", [](void *p) {
        Args *a = (Args *)p;
        swg_ctx *c = a->c;
        if (a->n == 0 || a->nu == 0) return;
        SWG_CUDA(cudaSetDevice(c->device));
        const u32 nu = a->nu;
        c->score_arena.reserve((size_t)nu * 16 + 1024); // small, context-owned (the scratch arena may hold the caller's data)
        u32 *fk = c->score_arena.take<u32>(nu);
        i64 *dl = c->score_arena.take<i64>(nu);
        SWG_CUDA(cudaMemcpyAsync(fk, a->fk, sizeof(u32) * nu, cudaMemcpyHostToDevice, c->stream));
        SWG_CUDA(cudaMemcpyAsync(dl, a->dl, sizeof(i64) * nu, cudaMemcpyHostToDevice, c->stream));
        u32 *ch = a->ch;
        launch_for<t_renumber>(a->n, c->stream, c->lc, [=] __device__(u32 i) {
            const u32 k = ch[i];
            if (k == 0) return;
            u32 lo = 0, hi = nu; // last run whose first chain number is <= k
            while (hi - lo > 1) { const u32 mid = (lo + hi) >> 1; if (fk[mid] <= k) lo = mid; else hi = mid; }
            ch[i] = (u32)((i64)k + dl[lo]);
        });
        SWG_CUDA(cudaStreamSynchronize(c->stream));
    }, &a);
}
// status bytes (0..3) -> 2 bits per record, 16 records per u32 (record i in bits 2*(i%16)); both DEVICE arrays
int swg_pack_status_device(swg_ctx *c, uint64_t n, const uint8_t *status_dev, uint32_t *packed_dev) {
    if (!c || (n && (!status_dev || !packed_dev)) || n >= 0x7FFFFFF0ull) return SWG_ERR_ARG;
    struct Args { swg_ctx *c; u32 n; const u8 *s; u32 *o; } a{c, (u32)n, status_dev, packed_dev};
    return guarded(c, "swg_pack_status_device", [](void *p) {
        Args *a = (Args *)p;
        swg_ctx *c = a->c;
        if (a->n == 0) return;
        SWG_CUDA(cudaSetDevice(c->device));
        const u32 n = a->n, nw = cdiv(n, 16);
        const u8 *st = a->s;
        u32 *out = a->o;
        launch_for<t_pack>(nw, c->stream, c->lc, [=] __device__(u32 w) {
            u32 v = 0;
            if ((u64)w * 16 + 16 <= n && ((size_t)(st + (size_t)w * 16) & 15) == 0) {
                const uint4 q = *reinterpret_cast<const uint4 *>(st + (size_t)w * 16);
                const u32 x[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
                for (int k = 0; k < 4; k++)
#pragma unroll
                    for (int b = 0; b < 4; b++) v |= ((x[k] >> (8 * b)) & 3u) << (2 * (4 * k + b));
            } else {
                for (u32 k = 0; k < 16 && (u64)w * 16 + k < n; k++) v |= ((u32)st[(size_t)w * 16 + k] & 3u) << (2 * k);
            }
            out[w] = v;
        });
        SWG_CUDA(cudaStreamSynchronize(c->stream));
    }, &a);
}

// ---- verification entry points: the f64 expressions of the path, evaluated on the device ------------------------
struct t_verify;
int swg_score_column(swg_ctx *c, uint64_t n, const double *identity, const uint32_t *qs, const uint32_t *qe, int scoring, double *out) {
    if (!c || (n && (!identity || !qs || !qe || !out)) || scoring < 0 || scoring > 4 || n >= 0x7FFFFFF0ull) return SWG_ERR_ARG;
    struct Args { swg_ctx *c; u32 n; const double *id; const u32 *qs, *qe; int scoring; double *out; } a{c, (u32)n, identity, qs, qe, scoring, out};
    return guarded(c, "swg_score_column", [](void *p) {
        Args *a = (Args *)p;
        swg_ctx *c = a->c;
        const u32 n = a->n;
        if (n == 0) return;
        SWG_CUDA(cudaSetDevice(c->device));
        c->arena.reserve((size_t)n * 24 + (1u << 20));
        double *id = c->arena.take<double>(n), *sc = c->arena.take<double>(n);
        u32 *qs = c->arena.take<u32>(n), *qe = c->arena.take<u32>(n);
        SWG_CUDA(cudaMemcpyAsync(id, a->id, (size_t)n * 8, cudaMemcpyHostToDevice, c->stream));
        SWG_CUDA(cudaMemcpyAsync(qs, a->qs, (size_t)n * 4, cudaMemcpyHostToDevice, c->stream));
        SWG_CUDA(cudaMemcpyAsync(qe, a->qe, (size_t)n * 4, cudaMemcpyHostToDevice, c->stream));
        const int scoring = a->scoring;
        const bool cuda_log = c->knobs.cuda_log;
        launch_for<t_verify>(n, c->stream, c->lc, [=] __device__(u32 i) { sc[i] = score_fn(scoring, id[i], qs[i], qe[i], cuda_log); });
        SWG_CUDA(cudaMemcpyAsync(a->out, sc, (size_t)n * 8, cudaMemcpyDeviceToHost, c->stream));
        SWG_CUDA(cudaStreamSynchronize(c->stream));
    }, &a);
}
int swg_chain_identity(swg_ctx *c, uint64_t n, const uint64_t *total_length, const uint64_t *sum_block, const uint64_t *sum_matches, double *out) {
    if (!c || (n && (!total_length || !sum_block || !sum_matches || !out)) || n >= 0x7FFFFFF0ull) return SWG_ERR_ARG;
    struct Args { swg_ctx *c; u32 n; const u64 *tl, *sb, *sm; double *out; } a{c, (u32)n, total_length, sum_block, sum_matches, out};
    return guarded(c, "swg_chain_identity", [](void *p) {
        Args *a = (Args *)p;
        swg_ctx *c = a->c;
        const u32 n = a->n;
        if (n == 0) return;
        SWG_CUDA(cudaSetDevice(c->device));
        c->arena.reserve((size_t)n * 32 + (1u << 20));
        u64 *tl = c->arena.take<u64>(n), *sb = c->arena.take<u64>(n), *sm = c->arena.take<u64>(n);
        double *w = c->arena.take<double>(n);
        SWG_CUDA(cudaMemcpyAsync(tl, a->tl, (size_t)n * 8, cudaMemcpyHostToDevice, c->stream));
        SWG_CUDA(cudaMemcpyAsync(sb, a->sb, (size_t)n * 8, cudaMemcpyHostToDevice, c->stream));
        SWG_CUDA(cudaMemcpyAsync(sm, a->sm, (size_t)n * 8, cudaMemcpyHostToDevice, c->stream));
        const bool cuda_log = c->knobs.cuda_log;
        launch_for<t_verify>(n, c->stream, c->lc, [=] __device__(u32 i) { w[i] = chain_identity_fn(tl[i], sb[i], sm[i], cuda_log); });
        SWG_CUDA(cudaMemcpyAsync(a->out, w, (size_t)n * 8, cudaMemcpyDeviceToHost, c->stream));
        SWG_CUDA(cudaStreamSynchronize(c->stream));
    }, &a);
}
int swg_log_matches_host(const swg_ctx *c) { return c ? (c->log_matches_host ? 1 : 0) : SWG_ERR_ARG; }
double swg_glibc_log_host(double x) { return glibc_log(x); }

// Tuning aid (not part of the public header): sort n pseudo-random (key,payload) pairs over `bits` key bits, `reps`
// times, and report the mean CUDA-event time of ONE one-sweep pass in *ms_per_pass.  Returns 0 and checks sortedness.
int swg__bench_sort(swg_ctx *c, uint64_t n, int bits, int reps, double *ms_per_pass, int *sorted_ok) {
    if (!c || !ms_per_pass || n == 0 || n >= 0x7FFFFFF0ull) return SWG_ERR_ARG;
    struct Args { swg_ctx *c; u32 n; int bits, reps; double *ms; int *ok; } a{c, (u32)n, bits, reps, ms_per_pass, sorted_ok};
    return guarded(c, "swg__bench_sort", [](void *p) {
        Args *a = (Args *)p;
        swg_ctx *c = a->c;
        SWG_CUDA(cudaSetDevice(c->device));
        const u32 n = a->n;
        c->arena.reserve((size_t)n * 40 + (64u << 20));
        u64 *src = c->arena.take<u64>(n), *k = c->arena.take<u64>(n), *k2 = c->arena.take<u64>(n);
        u32 *v = c->arena.take<u32>(n), *v2 = c->arena.take<u32>(n);
        u64 *bad = c->arena.take<u64>(1);
        const int bits = a->bits;
        launch_for<t_iota>(n, c->stream, c->lc, [=] __device__(u32 i) {
            u64 x = (u64)i * 0x9E3779B97F4A7C15ull + 0x7F4A7C15ull;
            x ^= x >> 29; x *= 0xBF58476D1CE4E5B9ull; x ^= x >> 32;
            src[i] = bits >= 64 ? x : (x & ((1ull << bits) - 1));
        });
        double total = 0;
        int passes = 1;
        for (int r = 0; r < a->reps; r++) {
            u64 *kk = k, *kk2 = k2;
            u32 *vv = v, *vv2 = v2;
            SWG_CUDA(cudaMemcpyAsync(kk, src, sizeof(u64) * n, cudaMemcpyDeviceToDevice, c->stream));
            launch_for<t_gather>(n, c->stream, c->lc, [=] __device__(u32 i) { vv[i] = i; });
            Arena::Mark mk = c->arena.mark();
            sort_pairs(c, kk, kk2, vv, vv2, n, bits, true);
            SWG_CUDA(cudaStreamSynchronize(c->stream));
            c->arena.rewind(mk);
            float ms = 0;
            SWG_CUDA(cudaEventElapsedTime(&ms, c->ev_sort[0], c->ev_sort[1]));
            total += ms;
            passes = c->sort_passes;
            if (r == a->reps - 1 && a->ok) {
                SWG_CUDA(cudaMemsetAsync(bad, 0, sizeof(u64), c->stream));
                const u64 *ks = kk;
                const u32 *vs = vv;
                launch_for<t_maxp>(n - 1, c->stream, c->lc, [=] __device__(u32 i) {
                    bool b = ks[i] > ks[i + 1] || (ks[i] == ks[i + 1] && vs[i] > vs[i + 1]) || src[vs[i]] != ks[i];
                    if (b) atomicAdd((unsigned long long *)bad, 1ull);
                });
                u64 hb = 1;
                SWG_CUDA(cudaMemcpyAsync(&hb, bad, sizeof(u64), cudaMemcpyDeviceToHost, c->stream));
                SWG_CUDA(cudaStreamSynchronize(c->stream));
                *a->ok = hb == 0;
            }
        }
        *a->ms = total / a->reps / passes;
    }, &a);
}

// The same for the packed sort (rs_sort_packed): *ms_per_pass = mean time of one packed-word pass (8 B read + 8 B written per
// element), *ms_total = the whole sort incl. histogram, pairs passes and the packing pass.  Checks that the result is the
// stable order of the full keys and that every word carries its key's high bits.
int swg__bench_sort_packed(swg_ctx *c, uint64_t n, int key_bits, int reps, double *ms_per_pass, double *ms_total, int *sorted_ok) {
    if (!c || !ms_per_pass || n == 0 || n >= 0x7FFFFFF0ull || key_bits > 64) return SWG_ERR_ARG;
    struct Args { swg_ctx *c; u32 n; int bits, reps; double *ms, *tot; int *ok; } a{c, (u32)n, key_bits, reps, ms_per_pass, ms_total, sorted_ok};
    return guarded(c, "swg__bench_sort_packed", [](void *p) {
        Args *a = (Args *)p;
        swg_ctx *c = a->c;
        SWG_CUDA(cudaSetDevice(c->device));
        const u32 n = a->n;
        c->arena.reserve((size_t)n * 40 + (64u << 20));
        u64 *src = c->arena.take<u64>(n), *k = c->arena.take<u64>(n), *k2 = c->arena.take<u64>(n);
        u32 *v = c->arena.take<u32>(n), *v2 = c->arena.take<u32>(n);
        u64 *bad = c->arena.take<u64>(1);
        const int bits = a->bits, ib = bits_for(n - 1);
        launch_for<t_iota>(n, c->stream, c->lc, [=] __device__(u32 i) {
            u64 x = (u64)i * 0x9E3779B97F4A7C15ull + 0x7F4A7C15ull;
            x ^= x >> 29; x *= 0xBF58476D1CE4E5B9ull; x ^= x >> 32;
            src[i] = bits >= 64 ? x : (x & ((1ull << bits) - 1));
        });
        double total = 0, whole = 0;
        PackedSort ps;
        for (int r = 0; r < a->reps; r++) {
            SWG_CUDA(cudaMemcpyAsync(k, src, sizeof(u64) * n, cudaMemcpyDeviceToDevice, c->stream));
            launch_for<t_gather>(n, c->stream, c->lc, [=] __device__(u32 i) { v[i] = i; });
            Arena::Mark mk = c->arena.mark();
            RadixSortPlan p = rs_plan(n, 0, bits);
            void *tmp = c->arena.take<char>(p.temp_bytes);
            SWG_CUDA(cudaEventRecord(c->ev[0], c->stream));
            ps = rs_sort_packed(n, bits, ib, k, k2, v, v2, tmp, p, c->stream, c->sm_count, c->lc, c->ev_sort[0], c->ev_sort[1]);
            SWG_CUDA(cudaEventRecord(c->ev[1], c->stream));
            SWG_CUDA(cudaStreamSynchronize(c->stream));
            c->arena.rewind(mk);
            float ms = 0, ms2 = 0;
            SWG_CUDA(cudaEventElapsedTime(&ms, c->ev_sort[0], c->ev_sort[1]));
            SWG_CUDA(cudaEventElapsedTime(&ms2, c->ev[0], c->ev[1]));
            total += ms / ps.timed_passes;
            whole += ms2;
        }
        if (a->ok) {
            SWG_CUDA(cudaMemsetAsync(bad, 0, sizeof(u64), c->stream));
            const u64 *w = ps.packed;
            const u64 mask = (1ull << ib) - 1;
            const int c0 = ps.c0;
            launch_for<t_maxp>(n, c->stream, c->lc, [=] __device__(u32 i) {
                const u32 a0 = (u32)(w[i] & mask);
                bool b = a0 >= n || (w[i] >> ib) != (src[a0 < n ? a0 : 0] >> c0);
                if (!b && i + 1 < n) {
                    const u32 a1 = (u32)(w[i + 1] & mask);
                    if (a1 < n) b = src[a0] > src[a1] || (src[a0] == src[a1] && a0 > a1);
                }
                if (b) atomicAdd((unsigned long long *)bad, 1ull);
            });
            u64 hb = 1;
            SWG_CUDA(cudaMemcpyAsync(&hb, bad, sizeof(u64), cudaMemcpyDeviceToHost, c->stream));
            SWG_CUDA(cudaStreamSynchronize(c->stream));
            *a->ok = hb == 0;
        }
        *a->ms = total / a->reps;
        if (a->tot) *a->tot = whole / a->reps;
    }, &a);
}

// ---- primitives: plane_sweep_exact.rs:268-461 -------------------------------------------------------
static int sweep_entry(swg_ctx *c, uint64_t n, const uint32_t *qs, const uint32_t *qe, const uint32_t *ts, const uint32_t *te,
                       const double *identity, uint64_t nq, uint64_t nt, double thr, int scoring, int axis, uint8_t *keep) {
    if (!c) return SWG_ERR_ARG;
    if (n && (!qs || !qe || !ts || !te || !identity || !keep)) { set_err(c, "NULL column"); return SWG_ERR_ARG; }
    if (scoring < 0 || scoring > 4 || n >= 0x7FFFFFF0ull) { set_err(c, "bad scoring / n"); return SWG_ERR_ARG; }
    for (uint64_t i = 0; i < n; i++)
        if (qe[i] < qs[i] || te[i] < ts[i]) { set_err(c, "interval with end < start"); return SWG_ERR_RANGE; }
    SweepArgs a{c, n, qs, qe, ts, te, identity, nq, nt, thr, scoring, axis, keep};
    return guarded(c, "swg_plane_sweep", do_sweep, &a);
}
int swg_plane_sweep_core(swg_ctx *c, uint64_t n, const uint32_t *begin, const uint32_t *end, const double *score, uint64_t max_to_keep,
                         double overlap_threshold, uint64_t *out_idx, uint64_t *n_out) {
    if (!c || !n_out || (n && (!begin || !end || !score || !out_idx)) || n >= 0x3FFFFFF0ull) return SWG_ERR_ARG;
    for (uint64_t i = 0; i < n; i++)
        if (end[i] < begin[i]) { set_err(c, "interval with end < begin"); return SWG_ERR_RANGE; }
    CoreArgs a{c, n, begin, end, score, max_to_keep, overlap_threshold, out_idx, n_out};
    return guarded(c, "swg_plane_sweep_core", do_sweep_core, &a);
}
int swg_plane_sweep_query(swg_ctx *c, uint64_t n, const uint32_t *qs, const uint32_t *qe, const uint32_t *ts, const uint32_t *te,
                          const double *identity, uint64_t n_keep, double thr, int scoring, uint8_t *keep) {
    return sweep_entry(c, n, qs, qe, ts, te, identity, n_keep, 0, thr, scoring, 0, keep);
}
int swg_plane_sweep_target(swg_ctx *c, uint64_t n, const uint32_t *qs, const uint32_t *qe, const uint32_t *ts, const uint32_t *te,
                           const double *identity, uint64_t n_keep, double thr, int scoring, uint8_t *keep) {
    return sweep_entry(c, n, qs, qe, ts, te, identity, 0, n_keep, thr, scoring, 1, keep);
}
int swg_plane_sweep_both(swg_ctx *c, uint64_t n, const uint32_t *qs, const uint32_t *qe, const uint32_t *ts, const uint32_t *te,
                         const double *identity, uint64_t nq, uint64_t nt, double thr, int scoring, uint8_t *keep) {
    return sweep_entry(c, n, qs, qe, ts, te, identity, nq, nt, thr, scoring, 2, keep);
}

// ---- file front end on the device (paf_device.cuh) ------------------------------------------------
int swg_filter_paf_host(swg_ctx *ctx, const swg_config *cfg, const char *in_path, const char *out_path, swg_stats *stats); // paf_io.cpp

// extract_metadata on the GPU; the table comes back as a host swg_paf (same accessors as swg_paf_parse).
swg_paf *swg_paf_parse_device(swg_ctx *c, const char *path) {
    if (!c) return nullptr;
    if (!path) { set_err(c, "swg_paf_parse_device: NULL path"); return nullptr; }
    swg_paf *p = new (std::nothrow) swg_paf();
    if (!p) return nullptr;
    {
        std::string err;
        if (!paf_open_text(path, p, &err)) { set_err(c, "swg_paf_parse_device: " + err); delete p; return nullptr; }
    }
    struct Args { swg_ctx *c; swg_paf *p; bool fallback; } a{c, p, false};
    const int rc = guarded(c, "swg_paf_parse_device", [](void *q) {
        Args *a = (Args *)q;
        swg_ctx *c = a->c;
        swg_paf *p = a->p;
        SWG_CUDA(cudaSetDevice(c->device));
        DevPaf dp;
        try { tokenize_device(c, PafText(*p), dp); } catch (const FrontEndFallback &) { a->fallback = true; return; }
        const size_t n = dp.n;
        p->n_lines = dp.n_lines;
        p->rank.resize(n); p->line_off.resize(n); p->line_len.resize(n);
        p->qid.resize(n); p->tid.resize(n); p->qs.resize(n); p->qe.resize(n); p->ts.resize(n); p->te.resize(n);
        p->blen.resize(n); p->matches.resize(n); p->identity.resize(n); p->strand.resize(n);
        p->names = dp.names; p->P = dp.hP; p->P2 = dp.hP2;
        if (n == 0) return;
        cudaStream_t st = c->stream;
        std::vector<u32> rank32;
        auto down = [&](void *dst, const void *src, size_t bytes) { SWG_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, st)); };
        if (dp.rank) { rank32.resize(n); down(rank32.data(), dp.rank, n * 4); }
        down(p->line_off.data(), dp.rec.off, n * 8); down(p->line_len.data(), dp.rec.len, n * 4);
        down(p->qid.data(), dp.qid, n * 4); down(p->tid.data(), dp.tid, n * 4);
        down(p->qs.data(), dp.rec.qs, n * 4); down(p->qe.data(), dp.rec.qe, n * 4);
        down(p->ts.data(), dp.rec.ts, n * 4); down(p->te.data(), dp.rec.te, n * 4);
        down(p->blen.data(), dp.rec.blen, n * 4); down(p->matches.data(), dp.rec.matches, n * 4);
        down(p->identity.data(), dp.rec.identity, n * 8); down(p->strand.data(), dp.rec.strand, n);
        SWG_CUDA(cudaStreamSynchronize(st));
        for (size_t r = 0; r < n; r++) p->rank[r] = dp.rank ? rank32[r] : r;
    }, &a);
    if (rc != SWG_OK) { delete p; return nullptr; }
    if (a.fallback) { // the device front end declined (oversize input, name hash collision): host front end
        delete p;
        char e[256];
        e[0] = 0;
        swg_paf *h = swg_paf_parse(path, e, sizeof e);
        if (!h) set_err(c, std::string("swg_paf_parse_device: ") + e);
        return h;
    }
    return p;
}

// PafFilter::filter_paf (src/paf_filter.rs:278-289) with the text tokenised, filtered and re-assembled on the GPU.
int swg_filter_paf(swg_ctx *c, const swg_config *cfg, const char *in_path, const char *out_path, swg_stats *stats) {
    if (!c || !cfg || !in_path || !out_path) return SWG_ERR_ARG;
    if (!check_cfg(c, cfg)) return SWG_ERR_ARG;
    c->knobs = read_knobs();
    if (c->knobs.paf_host_frontend) return swg_filter_paf_host(c, cfg, in_path, out_path, stats);
    swg_paf hp;
    if (const int orc = open_paf_text(c, "swg_filter_paf", in_path, &hp)) return orc;
    struct Args { swg_ctx *c; const swg_config *cfg; const swg_paf *hp; const char *out; swg_stats *stats; bool fallback; } a{c, cfg, &hp, out_path, stats, false};
    const int rc = guarded(c, "swg_filter_paf", [](void *q) {
        Args *a = (Args *)q;
        SWG_CUDA(cudaSetDevice(a->c->device));
        swg_stats local;
        try { filter_paf_device(a->c, *a->cfg, PafText(*a->hp), {a->out}, nullptr, local); } catch (const FrontEndFallback &) { a->fallback = true; return; }
        if (a->stats) *a->stats = local;
    }, &a);
    if (rc == SWG_OK && a.fallback) return swg_filter_paf_host(c, cfg, in_path, out_path, stats);
    return rc;
}

int swg_filter_paf_batch(swg_ctx *c, const swg_config *cfg, uint64_t n_files, const char *const *in_paths, const char *const *out_paths,
                         uint64_t *file_counts, swg_stats *stats) {
    if (!c) return SWG_ERR_ARG;
    if (!check_cfg(c, cfg)) return SWG_ERR_ARG;
    if (n_files == 0) {
        if (stats) std::memset(stats, 0, sizeof *stats);
        return SWG_OK;
    }
    const std::string who = "swg_filter_paf_batch: ";
    if (!in_paths || !out_paths) { set_err(c, who + "NULL path array"); return SWG_ERR_ARG; }
    if (n_files >= (1ull << 31)) { set_err(c, who + "too many files (must be < 2^31)"); return SWG_ERR_ARG; }
    {
        std::unordered_map<std::string, u64> seen;
        for (u64 k = 0; k < n_files; k++) {
            if (!in_paths[k] || !out_paths[k]) { set_err(c, who + "file " + std::to_string(k) + ": NULL path"); return SWG_ERR_ARG; }
            const auto ins = seen.emplace(out_paths[k], k);
            if (!ins.second) {
                set_err(c, who + "files " + std::to_string(ins.first->second) + " and " + std::to_string(k) + " have the same output path " + out_paths[k]);
                return SWG_ERR_ARG;
            }
        }
    }
    for (u64 k = 0; k < n_files; k++) { // every input opens before any output is created
        const int fd = open(in_paths[k], O_RDONLY);
        if (fd < 0) { set_err(c, who + "file " + std::to_string(k) + ": cannot open " + in_paths[k]); return SWG_ERR_IO; }
        close(fd);
    }
    PafBatchArgs a{c, cfg, n_files, in_paths, out_paths, file_counts, stats};
    return guarded(c, "swg_filter_paf_batch", do_filter_paf_batch, &a);
}

// calculate_ani_stats (src/main.rs:334-688) with the text tokenised and the per-pair sums accumulated on the GPU.
int swg_ani_stats(swg_ctx *c, const char *paf_path, int method, double percentile, int sort, double *ani50, uint64_t *n_pairs) {
    if (!c || !paf_path || !ani50) return SWG_ERR_ARG;
    if (method < SWG_ANI_ALL || method > SWG_ANI_NPERCENTILE || sort < SWG_NSORT_LENGTH || sort > SWG_NSORT_SCORE) {
        set_err(c, "swg_ani_stats: bad method / sort");
        return SWG_ERR_ARG;
    }
    std::string input = paf_path, tmp;
    if (method == SWG_ANI_ORTHOGONAL) { // best 1:1 mappings first (main.rs:346-383), then the plain statistic over the survivors
        swg_config cfg;
        swg_config_default(&cfg);
        cfg.min_block_length = 1000;
        cfg.mapping_filter_mode = SWG_ONE_TO_ONE; cfg.mapping_max_per_query = 1; cfg.mapping_max_per_target = 1;
        cfg.scaffold_filter_mode = SWG_ONE_TO_ONE; cfg.scaffold_max_per_query = 1; cfg.scaffold_max_per_target = 1;
        cfg.overlap_threshold = 0.95; cfg.scaffold_gap = 10000; cfg.min_scaffold_length = 0; cfg.scaffold_overlap_threshold = 0.95;
        cfg.scaffold_max_deviation = 0; cfg.scoring_function = SWG_SCORE_MATCHES; cfg.min_identity = 0.0; cfg.min_scaffold_identity = 0.0;
        cfg.keep_self = 0; cfg.scaffolds_only = 0;
        const char *td = getenv("TMPDIR");
        tmp = std::string(td && *td ? td : "/tmp") + "/swg_ani_XXXXXX";
        const int fd = mkstemp(&tmp[0]);
        if (fd < 0) { set_err(c, "swg_ani_stats: cannot create a temp file"); return SWG_ERR_IO; }
        close(fd);
        const int rc = swg_filter_paf(c, &cfg, paf_path, tmp.c_str(), nullptr);
        if (rc != SWG_OK) { unlink(tmp.c_str()); return rc; }
        input = tmp;
        method = SWG_ANI_ALL;
    }
    swg_paf hp;
    if (const int orc = open_paf_text(c, "swg_ani_stats", input.c_str(), &hp)) {
        if (!tmp.empty()) unlink(tmp.c_str());
        return orc;
    }
    struct Args { swg_ctx *c; const swg_paf *hp; int method; double pct; int sort; AniResult res; Declines d; } a{c, &hp, method, percentile, sort, {}, {}};
    int rc = guarded(c, "swg_ani_stats", [](void *q) {
        Args *a = (Args *)q;
        SWG_CUDA(cudaSetDevice(a->c->device));
        a->d.run([&] { a->res = ani_device(a->c, *a->hp, a->method, a->pct, a->sort); });
    }, &a);
    if (!tmp.empty()) unlink(tmp.c_str());
    if (rc == SWG_OK) rc = a.d.rc(c, "swg_ani_stats", "NaN among the sort keys or pair ANI values");
    if (rc != SWG_OK) return rc;
    *ani50 = a.res.ani50;
    if (n_pairs) *n_pairs = a.res.n_pairs;
    return SWG_OK;
}

// apply_tree_filter_to_paf (src/tree_filter.rs:205-283): tokenising, per-pair sums and the output on the GPU.
int swg_tree_filter_paf(swg_ctx *c, const char *in_path, const char *out_path, uint64_t k_nearest, uint64_t k_farthest,
                        double random_fraction, uint64_t *n_kept, uint64_t *n_pairs_selected) {
    if (!c || !in_path || !out_path) return SWG_ERR_ARG;
    swg_paf hp;
    if (const int orc = open_paf_text(c, "swg_tree_filter_paf", in_path, &hp)) return orc;
    struct Args { swg_ctx *c; const swg_paf *hp; const char *out; u64 kn, kf; double rf; TreeResult res; Declines d; } a{c, &hp, out_path, k_nearest, k_farthest, random_fraction, {}, {}};
    int rc = guarded(c, "swg_tree_filter_paf", [](void *q) {
        Args *a = (Args *)q;
        SWG_CUDA(cudaSetDevice(a->c->device));
        a->d.run([&] { a->res = tree_filter_device(a->c, *a->hp, a->out, a->kn, a->kf, a->rf); });
    }, &a);
    if (rc == SWG_OK) rc = a.d.rc(c, "swg_tree_filter_paf", "NaN identity");
    if (rc != SWG_OK) return rc;
    if (n_kept) *n_kept = a.res.n_kept;
    if (n_pairs_selected) *n_pairs_selected = a.res.n_selected;
    return SWG_OK;
}

} // extern "C"

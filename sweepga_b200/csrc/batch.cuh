// batch.cuh — swg_filter_batch: many independent mapping tables filtered by ONE run of the pipeline (DESIGN §6a).
//
// The K tables are laid end to end on the device with disjoint ids: sequence ids shifted by the running n_seq, genome-prefix
// ids (P, P2) by the running genome count.  Every grouping of apply_filters stays inside one table then, and chains are
// numbered by the input index of their unit's first stage-1 record, so table k's chains are one consecutive run of the
// union's numbering.  The union runs through run_filter_exact unchanged; afterwards one pass subtracts every table's chain
// offset and tallies its counts.  Per call: one gathered upload (one DMA per 8 MiB piece, whatever K is), three kernels of
// our own, one scattered download.
#pragma once

namespace swg {

// per-table layout of the union (device copy next to the record and sequence offsets)
struct BatchTable {
    u64 id_off;  // byte offset of the table's raw id columns in the union's id buffers
    u32 n_seq;   // the table's own n_seq: a local id >= n_seq becomes NONE32 (a range error once it reaches k_prefilter)
    u32 seq_off; // first union sequence id of the table
    u32 goff;    // added to the table's P and P2 ids
    u32 id16;    // 1: 16-bit id columns
    u32 derive;  // 1: no identity column — k_batch_ids writes matches / max(block_length, 1) into the union's
    u32 pad;
};
constexpr u32 BATCH_SMEM_TABLES = 8192; // record offsets held in shared memory up to this many tables (32 KB)

// table of union position i: the largest k < K with off[k] <= i (off[0] = 0 <= i < off[K]; empty tables are skipped)
__device__ __forceinline__ u32 batch_table_of(const u32 *off, u32 K, u32 i) { return file_at<u32>(off, K, i); }
// the K + 1 record offsets in shared memory when they fit, else read from global memory
__device__ __forceinline__ const u32 *batch_offsets(const u32 *rec_off, u32 K, u32 *s_off) {
    if (K + 1 > BATCH_SMEM_TABLES) return rec_off;
    for (u32 k = threadIdx.x; k <= K; k += blockDim.x) s_off[k] = rec_off[k];
    __syncthreads();
    return s_off;
}

// Union ids, one pass: records [0, N) get their 32-bit union query / target ids (16-bit columns widened on the way) and, for
// tables without an identity column, the parser's identity (rec_identity's division, so the same bits); sequences [N, N + S)
// get their table's genome offset added to P and P2.  Grid-stride over a fixed grid, so the offsets are loaded once per CTA.
__global__ void __launch_bounds__(256) k_batch_ids(u32 N, u32 S, u32 K, const u32 *__restrict__ rec_off, const u32 *__restrict__ seq_off,
                                                   const BatchTable *__restrict__ tab, const char *__restrict__ qraw,
                                                   const char *__restrict__ traw, u32 *__restrict__ qid, u32 *__restrict__ tid,
                                                   const u32 *__restrict__ blen, const u32 *__restrict__ matches, double *__restrict__ identity,
                                                   u32 *__restrict__ P, u32 *__restrict__ P2) {
    extern __shared__ u32 s_off[];
    const u32 *off = batch_offsets(rec_off, K, s_off);
    const u32 stride = gridDim.x * blockDim.x;
    for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < N; i += stride) {
        const u32 k = batch_table_of(off, K, i);
        const BatchTable t = tab[k];
        const u32 j = i - off[k];
        u32 q, r;
        if (t.id16) {
            q = reinterpret_cast<const u16 *>(qraw + t.id_off)[j];
            r = reinterpret_cast<const u16 *>(traw + t.id_off)[j];
        } else {
            q = reinterpret_cast<const u32 *>(qraw + t.id_off)[j];
            r = reinterpret_cast<const u32 *>(traw + t.id_off)[j];
        }
        qid[i] = q < t.n_seq ? q + t.seq_off : NONE32;
        tid[i] = r < t.n_seq ? r + t.seq_off : NONE32;
        if (t.derive && identity) {
            const u32 b = blen[i];
            identity[i] = __ddiv_rn((double)matches[i], (double)(b > 1 ? b : 1));
        }
    }
    for (u32 s = blockIdx.x * blockDim.x + threadIdx.x; s < S; s += stride) {
        const u32 g = tab[batch_table_of(seq_off, K, s)].goff;
        P[s] += g;
        P2[s] += g;
    }
}

// chain_off[k] = kept chains of tables 0..k-1 = chains whose unit starts before record rec_off[k] (key_a, the input index of
// the unit's first stage-1 record, is nondecreasing in chain order); CHAINS_KEPT of table k = chain_off[k + 1] - chain_off[k].
__global__ void __launch_bounds__(256) k_batch_chain_off(u32 K, const u32 *__restrict__ rec_off, const u32 *__restrict__ key_a, u32 n_chains,
                                                         u32 *__restrict__ chain_off, u64 *__restrict__ counts) {
    const u32 k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k > K) return;
    auto lower = [&](u32 x) {
        u32 lo = 0, hi = n_chains;
        while (lo < hi) {
            const u32 mid = (lo + hi) >> 1;
            if (key_a[mid] < x) lo = mid + 1;
            else hi = mid;
        }
        return lo;
    };
    const u32 a = lower(rec_off[k]);
    chain_off[k] = a;
    if (k < K) counts[(u64)k * SWG_TC_COUNT + SWG_TC_CHAINS_KEPT] = lower(rec_off[k + 1]) - a;
}

// Per record: chain numbers renumbered per table (chain_id -= chain_off[table]), and the table's STAGE1 / KEPT / SCAFFOLD /
// RESCUED counts.  Every warp walks one contiguous span 32 records at a time with a segmented scan over its lanes; a run of one
// table is carried from step to step and flushed with one atomic per counter only where the table changes (and once at the
// end of the span), so many tiny tables cost an atomic per table boundary, not per record.
__global__ void __launch_bounds__(256) k_batch_finish(u32 N, u32 K, const u32 *__restrict__ rec_off, const u32 *__restrict__ chain_off,
                                                      const u8 *__restrict__ flags, const u8 *__restrict__ status, u32 *__restrict__ chain_id,
                                                      u64 *__restrict__ counts) {
    extern __shared__ u32 s_off[];
    const u32 *off = batch_offsets(rec_off, K, s_off);
    const u32 full = 0xFFFFFFFFu, lane = lane_id();
    const u32 warps = gridDim.x * (blockDim.x >> 5), w = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const u32 span = (u32)(((((u64)N + warps - 1) / warps) + 31) & ~31ull);
    const u64 b0 = (u64)w * span;
    if (b0 >= N) return;
    const u32 b1 = (u32)(b0 + span < N ? b0 + span : N);
    u32 ctab = NONE32, cv[4] = {0, 0, 0, 0}; // the carried run (warp-uniform)
    auto flush = [&](u32 t, const u32 (&v)[4]) {
        for (int c = 0; c < 4; c++)
            if (v[c]) atomicAdd((unsigned long long *)&counts[(u64)t * SWG_TC_COUNT + c], (unsigned long long)v[c]);
    };
    for (u32 base = (u32)b0; base < b1; base += 32) {
        const u32 i = base + lane;
        const bool in = i < b1;
        u32 t = NONE32, v[4] = {0, 0, 0, 0};
        if (in) {
            t = batch_table_of(off, K, i);
            const u8 s = status[i];
            v[0] = (flags[i] & F_ALIVE) ? 1u : 0u;
            v[1] = s != 0;
            v[2] = s == 1;
            v[3] = s == 2;
            const u32 ch = chain_id[i];
            if (ch) chain_id[i] = ch - chain_off[t];
        }
        // the carried run continues into lane 0's table, or is flushed
        const u32 t0 = __shfl_sync(full, t, 0);
        if (ctab != NONE32 && ctab != t0) {
            if (lane == 0) flush(ctab, cv);
            cv[0] = cv[1] = cv[2] = cv[3] = 0;
        }
        if (lane == 0)
            for (int c = 0; c < 4; c++) v[c] += cv[c];
        // inclusive segmented scan (segments are contiguous lane ranges of one table)
#pragma unroll
        for (u32 d = 1; d < 32; d <<= 1) {
            const u32 tu = __shfl_up_sync(full, t, d);
#pragma unroll
            for (int c = 0; c < 4; c++) {
                const u32 vu = __shfl_up_sync(full, v[c], d);
                if (lane >= d && tu == t) v[c] += vu;
            }
        }
        const u32 tn = __shfl_down_sync(full, t, 1);
        if (in && lane < 31 && tn != t) flush(t, v); // a run that ends inside this step
        ctab = __shfl_sync(full, t, 31);
        for (int c = 0; c < 4; c++) cv[c] = __shfl_sync(full, v[c], 31);
    }
    if (lane == 0 && ctab != NONE32) flush(ctab, cv);
}

// ---- host side -----------------------------------------------------------------------------------------------------------
struct BatchArgs {
    swg_ctx *c; const swg_config *cfg; u64 K; const swg_mappings *in; swg_result *out; u64 *counts; swg_stats *stats;
};

static void do_filter_batch(void *p) {
    BatchArgs *a = (BatchArgs *)p;
    swg_ctx *c = a->c;
    const u32 K = (u32)a->K;
    const swg_mappings *in = a->in;
    SWG_CUDA(cudaSetDevice(c->device));
    // the union's chain keys describe no table's numbering: the context reports no chains after this call, whatever happens
    struct ForgetChains {
        swg_ctx *c;
        ~ForgetChains() { c->last_n_chains = 0; c->last_keyA = c->last_keyB = nullptr; c->last_flags = nullptr; }
    } forget{c};
    swg_stats S;
    std::memset(&S, 0, sizeof S);
    if (a->counts) std::memset(a->counts, 0, sizeof(u64) * SWG_TC_COUNT * (size_t)K);

    // ---- layout of the union (host) ----------------------------------------------------------------------------------------
    std::vector<u32> rec_off(K + 1), seq_off(K + 1);
    std::vector<BatchTable> tab(K);
    u64 N = 0, S_seq = 0, G = 0, id_bytes = 0;
    bool any_identity = false;
    for (u32 k = 0; k < K; k++) {
        const swg_mappings &m = in[k];
        rec_off[k] = (u32)N;
        seq_off[k] = (u32)S_seq;
        BatchTable &t = tab[k];
        std::memset(&t, 0, sizeof t);
        t.seq_off = (u32)S_seq;
        t.id_off = id_bytes;
        if (m.n == 0) continue; // contributes nothing, not even its sequences
        t.n_seq = m.n_seq;
        t.id16 = m.query_id == nullptr;
        t.derive = m.identity == nullptr;
        any_identity |= m.identity != nullptr;
        // run_filter's check of the prefix ids, per table (in the union a too-large id could still fall below the total)
        u32 mx = 0;
        for (u32 s = 0; s < m.n_seq; s++) mx = std::max(mx, std::max(m.seq_genome_id[s], m.seq_genome2_id[s]));
        if (mx >= m.n_seq) throw RangeError{"table " + std::to_string(k) + ": genome prefix id >= n_seq (prefix ids must be dense)"};
        t.goff = (u32)G;
        G += (u64)mx + 1;
        N += m.n;
        S_seq += m.n_seq;
        id_bytes += (m.n * (t.id16 ? 2 : 4) + 3) & ~(u64)3; // every table's id slice starts 4-byte aligned
    }
    rec_off[K] = (u32)N;
    seq_off[K] = (u32)S_seq;
    S.n_input = N;
    const u64 launches0 = c->lc.n;
    if (N == 0) {
        if (a->stats) *a->stats = S;
        return;
    }
    bool any_score = false;
    for (u32 k = 0; k < K; k++) any_score |= in[k].n && in[k].score;

    // ---- device layout (context-owned arena: run_filter rewinds c->arena, the prefetch slots own theirs) ----------------------
    const size_t meta_bytes = sizeof(u32) * 2 * (K + 1) + sizeof(BatchTable) * K;
    c->batch.reserve(id_bytes * 2 + N * (6 * 4 + (any_identity ? 8 : 0) + (any_score ? 8 : 0) + 1 + 8 + 5) + S_seq * 8 + meta_bytes +
                     (size_t)K * (4 + 8 * SWG_TC_COUNT) + 32 * 256);
    Arena &B = c->batch;
    char *qraw = B.take<char>(id_bytes), *traw = B.take<char>(id_bytes);
    u32 *qs = B.take<u32>(N), *qe = B.take<u32>(N), *ts = B.take<u32>(N), *te = B.take<u32>(N), *bl = B.take<u32>(N), *mt = B.take<u32>(N);
    double *idy = any_identity ? B.take<double>(N) : nullptr;
    double *score = any_score ? B.take<double>(N) : nullptr;
    u8 *strand = B.take<u8>(N);
    u32 *P = B.take<u32>(S_seq), *P2 = B.take<u32>(S_seq);
    char *meta = B.take<char>(meta_bytes);
    u32 *d_rec_off = reinterpret_cast<u32 *>(meta), *d_seq_off = d_rec_off + (K + 1);
    BatchTable *d_tab = reinterpret_cast<BatchTable *>(meta + sizeof(u32) * 2 * (K + 1)); // 8-byte aligned: K + 1 u32 twice
    u32 *qid = B.take<u32>(N), *tid = B.take<u32>(N);
    u8 *status = B.take<u8>(N);
    u32 *chain_id = B.take<u32>(N), *chain_off = B.take<u32>(K + 1);
    u64 *counts = B.take<u64>((size_t)K * SWG_TC_COUNT);

    // ---- upload: one column = one device range fed by K host slices ------------------------------------------------------------
    std::vector<char> hmeta(meta_bytes);
    std::memcpy(hmeta.data(), rec_off.data(), sizeof(u32) * (K + 1));
    std::memcpy(hmeta.data() + sizeof(u32) * (K + 1), seq_off.data(), sizeof(u32) * (K + 1));
    std::memcpy(hmeta.data() + sizeof(u32) * 2 * (K + 1), tab.data(), sizeof(BatchTable) * K);
    std::vector<PinCol> cols;
    auto column = [&](void *dev, size_t bytes, auto host_of, size_t elem, bool per_seq) {
        PinCol col{(char *)dev, bytes, {}};
        for (u32 k = 0; k < K; k++) {
            const swg_mappings &m = in[k];
            const char *h = (const char *)host_of(m);
            const size_t cnt = per_seq ? m.n_seq : m.n;
            if (m.n == 0 || !h) continue;
            col.segs.push_back(PinSeg{(char *)h, (size_t)(per_seq ? seq_off[k] : rec_off[k]) * elem, cnt * elem});
        }
        cols.push_back(std::move(col));
    };
    for (int side = 0; side < 2; side++) {
        PinCol col{side ? traw : qraw, id_bytes, {}};
        for (u32 k = 0; k < K; k++) {
            const swg_mappings &m = in[k];
            if (m.n == 0) continue;
            const void *h = tab[k].id16 ? (const void *)(side ? m.target_id16 : m.query_id16) : (const void *)(side ? m.target_id : m.query_id);
            col.segs.push_back(PinSeg{(char *)h, tab[k].id_off, m.n * (tab[k].id16 ? 2 : 4)});
        }
        cols.push_back(std::move(col));
    }
    column(qs, N * 4, [](const swg_mappings &m) { return m.query_start; }, 4, false);
    column(qe, N * 4, [](const swg_mappings &m) { return m.query_end; }, 4, false);
    column(ts, N * 4, [](const swg_mappings &m) { return m.target_start; }, 4, false);
    column(te, N * 4, [](const swg_mappings &m) { return m.target_end; }, 4, false);
    column(bl, N * 4, [](const swg_mappings &m) { return m.block_length; }, 4, false);
    column(mt, N * 4, [](const swg_mappings &m) { return m.matches; }, 4, false);
    if (idy) column(idy, N * 8, [](const swg_mappings &m) { return m.identity; }, 8, false); // tables without one: k_batch_ids
    if (score) column(score, N * 8, [](const swg_mappings &m) { return m.score; }, 8, false);
    column(strand, N, [](const swg_mappings &m) { return m.strand; }, 1, false);
    column(P, S_seq * 4, [](const swg_mappings &m) { return m.seq_genome_id; }, 4, true);
    column(P2, S_seq * 4, [](const swg_mappings &m) { return m.seq_genome2_id; }, 4, true);
    cols.push_back(PinCol{meta, meta_bytes, {PinSeg{hmeta.data(), 0, meta_bytes}}});
    size_t h2d = 0;
    for (const PinCol &col : cols) h2d += col.bytes;

    cudaStream_t st = c->stream;
    SWG_CUDA(cudaEventRecord(c->ev[0], st));
    SWG_CUDA(cudaStreamWaitEvent(c->copy_stream, c->ev[0], 0));
    staged_h2d_cols(c, cols);
    SWG_CUDA(cudaEventRecord(c->ev_copy[0], c->copy_stream));
    SWG_CUDA(cudaStreamWaitEvent(st, c->ev_copy[0], 0));
    SWG_CUDA(cudaEventRecord(c->ev[1], st));

    // ---- union ids, the filter, per-table renumbering and counts -------------------------------------------------------------
    const u32 grid = (u32)c->sm_count * 8;
    const size_t smem = K + 1 <= BATCH_SMEM_TABLES ? sizeof(u32) * (K + 1) : 0;
    k_batch_ids<<<grid, 256, smem, st>>>((u32)N, (u32)S_seq, K, d_rec_off, d_seq_off, d_tab, qraw, traw, qid, tid, bl, mt, idy, P, P2);
    c->lc.n++;
    DevIn u;
    u.qid = qid; u.tid = tid; u.qs = qs; u.qe = qe; u.ts = ts; u.te = te; u.blen = bl; u.matches = mt;
    u.identity = idy; u.strand = strand; u.score = score; u.P = P; u.P2 = P2; u.n = (u32)N; u.n_seq = (u32)S_seq;
    swg_stats F;
    run_filter_exact(c, *a->cfg, u, status, chain_id, &F, nullptr, nullptr);
    // c->last_flags lives in the scratch arena: read it before anything else takes from there
    SWG_CUDA(cudaMemsetAsync(counts, 0, sizeof(u64) * SWG_TC_COUNT * (size_t)K, st));
    k_batch_chain_off<<<cdiv(K + 1, 256), 256, 0, st>>>(K, d_rec_off, c->last_keyA, c->last_keyA ? (u32)c->last_n_chains : 0u, chain_off, counts);
    k_batch_finish<<<grid, 256, smem, st>>>((u32)N, K, d_rec_off, chain_off, c->last_flags, status, chain_id, counts);
    c->lc.n += 2;
    SWG_CUDA(cudaEventRecord(c->ev[2], st));

    // ---- download: one DMA per piece, the host team scatters into the K caller arrays ---------------------------------------
    std::vector<PinCol> outs(2);
    outs[0] = PinCol{(char *)status, N, {}};
    outs[1] = PinCol{(char *)chain_id, N * 4, {}};
    for (u32 k = 0; k < K; k++) {
        if (in[k].n == 0) continue;
        outs[0].segs.push_back(PinSeg{(char *)a->out[k].status, rec_off[k], in[k].n});
        outs[1].segs.push_back(PinSeg{(char *)a->out[k].chain_id, (size_t)rec_off[k] * 4, in[k].n * 4});
    }
    if (a->counts) outs.push_back(PinCol{(char *)counts, sizeof(u64) * SWG_TC_COUNT * (size_t)K, {PinSeg{(char *)a->counts, 0, sizeof(u64) * SWG_TC_COUNT * (size_t)K}}});
    size_t d2h = 0;
    for (const PinCol &col : outs) d2h += col.bytes;
    SWG_CUDA(cudaStreamWaitEvent(c->copy_stream, c->ev[2], 0));
    staged_d2h_cols(c, outs);
    SWG_CUDA(cudaEventRecord(c->ev_copy[1], c->copy_stream));
    SWG_CUDA(cudaStreamWaitEvent(st, c->ev_copy[1], 0));
    SWG_CUDA(cudaEventRecord(c->ev[3], st));
    SWG_CUDA(cudaStreamSynchronize(st));

    float m0 = 0, m1 = 0, m2 = 0;
    SWG_CUDA(cudaEventElapsedTime(&m0, c->ev[0], c->ev[1]));
    SWG_CUDA(cudaEventElapsedTime(&m1, c->ev[1], c->ev[2]));
    SWG_CUDA(cudaEventElapsedTime(&m2, c->ev[2], c->ev[3]));
    F.ms_h2d = m0; F.ms_device = m1; F.ms_d2h = m2;
    F.h2d_bytes = h2d;
    F.d2h_bytes = d2h;
    F.gpu_launches = c->lc.n - launches0;
    if (a->stats) *a->stats = F;
}

// ---- many PAF files in one call (swg_filter_paf_batch, DESIGN §6b) ----------------------------------------------------------
// Consecutive files form one union (PafText): one upload, one newline scan, one parse, one name table with a namespace per
// file, one run of the filter, the per-file renumbering above, and one writer that sends every piece of the union's output to
// the files it overlaps.  Launches grow with the data, not with the number of files.

static void add_stats(swg_stats &a, const swg_stats &b) {
    a.n_input += b.n_input; a.n_stage1 += b.n_stage1; a.n_after_sweep += b.n_after_sweep; a.n_chains += b.n_chains;
    a.n_chains_after_mass += b.n_chains_after_mass; a.n_chains_kept += b.n_chains_kept; a.n_anchors += b.n_anchors;
    a.n_rescued += b.n_rescued; a.n_kept += b.n_kept; a.score_near_ties += b.score_near_ties; a.gpu_launches += b.gpu_launches;
    a.ms_h2d += b.ms_h2d; a.ms_device += b.ms_device; a.ms_d2h += b.ms_d2h; a.ms_sort_passes += b.ms_sort_passes;
    a.n_sort_passes += b.n_sort_passes; a.n_sort_pairs += b.n_sort_pairs; a.ms_tokenize += b.ms_tokenize; a.ms_write += b.ms_write;
    a.exact_rerank |= b.exact_rerank; a.h2d_bytes += b.h2d_bytes; a.d2h_bytes += b.d2h_bytes; a.n_dirty_groups += b.n_dirty_groups;
    a.ms_prefilter += b.ms_prefilter; a.n_unsorted_groups += b.n_unsorted_groups;
    if (b.sort_bytes_per_pair) a.sort_bytes_per_pair = b.sort_bytes_per_pair;
    if (b.prefilter_bytes_per_record) a.prefilter_bytes_per_record = b.prefilter_bytes_per_record;
}

// A text (one file, or a union of files) through the device front end, the filter and the writer; out_paths[k] receives the
// output of file k.  counts (K rows of SWG_TC_COUNT, or nullptr for a plain swg_filter_paf): the union's chains are renumbered
// per file and every file's counts tallied.  FrontEndFallback: the device declines the text, and nothing was written.
static void filter_paf_device(swg_ctx *c, const swg_config &cfg, const PafText &tx, const std::vector<const char *> &out_paths, u64 *counts,
                              swg_stats &S) {
    cudaStream_t st = c->stream;
    const u64 launches0 = c->lc.n;
    DevPaf dp;
    tokenize_device(c, tx, dp);
    std::memset(&S, 0, sizeof S);
    const u32 n = dp.n, K = tx.K();
    u8 *status = c->io.take<u8>(std::max<u32>(n, 1));
    u32 *chain = c->io.take<u32>(std::max<u32>(n, 1));
    u64 *d_counts = counts ? c->io.take<u64>((size_t)K * SWG_TC_COUNT) : nullptr;
    if (counts) SWG_CUDA(cudaMemsetAsync(d_counts, 0, sizeof(u64) * SWG_TC_COUNT * (size_t)K, st));
    if (n) {
        SWG_CUDA(cudaEventRecord(c->ev[1], st));
        run_filter_exact(c, cfg, devin_of(dp), status, chain, &S, nullptr, nullptr);
        if (counts) { // c->last_flags lives in the scratch arena, which write_device takes from: tally first
            u32 *rec_off = dp.rec_off;
            if (!rec_off) {
                rec_off = c->io.take<u32>(K + 1);
                SWG_CUDA(cudaMemcpyAsync(rec_off, dp.file_rec.data(), sizeof(u32) * (K + 1), cudaMemcpyHostToDevice, st));
            }
            u32 *chain_off = c->io.take<u32>(K + 1);
            const size_t smem = K + 1 <= BATCH_SMEM_TABLES ? sizeof(u32) * (K + 1) : 0;
            k_batch_chain_off<<<cdiv(K + 1, 256), 256, 0, st>>>(K, rec_off, c->last_keyA, c->last_keyA ? (u32)c->last_n_chains : 0u, chain_off, d_counts);
            k_batch_finish<<<(u32)c->sm_count * 8, 256, smem, st>>>(n, K, rec_off, chain_off, c->last_flags, status, chain, d_counts);
            c->lc.n += 2;
        }
        SWG_CUDA(cudaEventRecord(c->ev[2], st));
        SWG_CUDA(cudaStreamSynchronize(st));
        float ms = 0;
        SWG_CUDA(cudaEventElapsedTime(&ms, c->ev[1], c->ev[2]));
        S.ms_device = ms;
    }
    if (counts) {
        SWG_CUDA(cudaMemcpyAsync(counts, d_counts, sizeof(u64) * SWG_TC_COUNT * (size_t)K, cudaMemcpyDeviceToHost, st));
        SWG_CUDA(cudaStreamSynchronize(st));
    }
    const auto t0 = std::chrono::steady_clock::now();
    write_device(c, dp, status, chain, out_paths);
    S.ms_write = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    S.ms_h2d = dp.ms_upload;
    S.ms_tokenize = dp.ms_tokenize;
    S.gpu_launches = c->lc.n - launches0;
}

struct PafBatchArgs {
    swg_ctx *c; const swg_config *cfg; u64 K; const char *const *in; const char *const *out; u64 *counts; swg_stats *stats;
};

static std::string file_name(const PafBatchArgs &a, u64 k) { return "file " + std::to_string(k) + " (" + a.in[k] + ")"; }

// The files [first, first + K) on the host route: swg_paf_parse per file, one swg_filter_batch, swg_paf_write per file.
static void filter_paf_host_group(const PafBatchArgs &a, u64 first, u32 K, u64 *counts, swg_stats &S) {
    std::vector<swg_paf *> ps(K, nullptr);
    struct Free { std::vector<swg_paf *> &p; ~Free() { for (swg_paf *x : p) swg_paf_free(x); } } free_all{ps};
    std::vector<swg_mappings> maps(K);
    for (u32 k = 0; k < K; k++) {
        char err[256];
        err[0] = 0;
        ps[k] = swg_paf_parse(a.in[first + k], err, sizeof err);
        if (!ps[k]) throw IoError{file_name(a, first + k) + ": " + err};
        swg_paf_view(ps[k], &maps[k]);
    }
    std::vector<std::vector<u8>> status(K);
    std::vector<std::vector<u32>> chain(K);
    std::vector<swg_result> res(K);
    for (u32 k = 0; k < K; k++) {
        status[k].resize(maps[k].n);
        chain[k].resize(maps[k].n);
        res[k] = swg_result{status[k].data(), chain[k].data()};
    }
    BatchArgs ba{a.c, a.cfg, K, maps.data(), res.data(), counts, &S};
    do_filter_batch(&ba);
    const auto t0 = std::chrono::steady_clock::now();
    for (u32 k = 0; k < K; k++)
        if (swg_paf_write(ps[k], a.out[first + k], status[k].data(), chain[k].data()) != SWG_OK)
            throw IoError{file_name(a, first + k) + ": cannot write " + a.out[first + k]};
    S.ms_write = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
}

// One group: the files [first, first + group.size()), already open.  The device route, or the host route when the device
// declines (or SWG_PAF_FRONTEND=host).  A union with more lines than mem_budget allows is split, and its two halves are
// filtered one after the other.  A range error of a union is located by filtering its files one at a time: the first file
// that fails alone fails the call, named; when every file passes alone, their results are the call's.
static void filter_paf_group(const PafBatchArgs &a, u64 first, std::vector<std::unique_ptr<swg_paf>> &group, u64 mem_budget, swg_stats &S) {
    swg_ctx *c = a.c;
    const u32 K = (u32)group.size();
    std::vector<u64> counts((size_t)K * SWG_TC_COUNT);
    swg_stats gs;
    std::memset(&gs, 0, sizeof gs);
    bool split = false, one_by_one = false;
    try {
        bool host = c->knobs.paf_host_frontend;
        if (!host) {
            std::vector<const swg_paf *> files;
            for (auto &p : group) files.push_back(p.get());
            PafText tx(files);
            tx.mem_budget = mem_budget;
            try {
                filter_paf_device(c, *a.cfg, tx, std::vector<const char *>(a.out + first, a.out + first + K), counts.data(), gs);
            } catch (const FrontEndFallback &) { host = true; } catch (const GroupTooLarge &) { split = true; }
        }
        if (host) filter_paf_host_group(a, first, K, counts.data(), gs);
    } catch (const RangeError &e) {
        if (K == 1) throw RangeError{file_name(a, first) + ": " + e.msg};
        one_by_one = true;
    }
    if (split || one_by_one) { // nothing of this union was written; its parts are filtered instead
        const u32 parts = split ? 2 : K;
        for (u32 p = 0; p < parts; p++) {
            const u32 k0 = (u32)((u64)K * p / parts), k1 = (u32)((u64)K * (p + 1) / parts);
            std::vector<std::unique_ptr<swg_paf>> part;
            for (u32 k = k0; k < k1; k++) part.push_back(std::move(group[k]));
            filter_paf_group(a, first + k0, part, mem_budget, S);
        }
        return;
    }
    if (a.counts) std::memcpy(a.counts + first * SWG_TC_COUNT, counts.data(), sizeof(u64) * counts.size());
    add_stats(S, gs);
}

static size_t arena_bytes(const Arena &A) {
    size_t b = 0;
    for (const auto &blk : A.blocks) b += blk.cap;
    return b;
}

static void do_filter_paf_batch(void *p) {
    const PafBatchArgs &a = *(const PafBatchArgs *)p;
    swg_ctx *c = a.c;
    SWG_CUDA(cudaSetDevice(c->device));
    struct ForgetChains { // as after swg_filter_batch: the union's chain keys describe no file's numbering
        swg_ctx *c;
        ~ForgetChains() { c->last_n_chains = 0; c->last_keyA = c->last_keyB = nullptr; c->last_flags = nullptr; }
    } forget{c};
    swg_stats S;
    std::memset(&S, 0, sizeof S);
    if (a.counts) std::memset(a.counts, 0, sizeof(u64) * SWG_TC_COUNT * (size_t)a.K);
    // limits of one group: those of a single file, the device memory free at the start of the call (plus what the context's
    // reusable arenas hold), and open files: a group holds its inputs and its outputs open
    size_t free_b = 0, total_b = 0;
    SWG_CUDA(cudaMemGetInfo(&free_b, &total_b));
    const u64 mem_budget = c->knobs.paf_batch_memory ? c->knobs.paf_batch_memory : (u64)free_b + arena_bytes(c->io) + arena_bytes(c->arena);
    const u64 byte_cap = std::min<u64>((1ull << 36) - 1, c->knobs.paf_batch_bytes ? c->knobs.paf_batch_bytes : ~0ull);
    u64 file_cap = 1ull << 31;
    {
        struct rlimit rl;
        if (getrlimit(RLIMIT_NOFILE, &rl) == 0 && rl.rlim_cur != RLIM_INFINITY) file_cap = std::max<u64>(1, ((u64)rl.rlim_cur - std::min<u64>(rl.rlim_cur, 64)) / 2);
    }
    std::vector<std::unique_ptr<swg_paf>> group;
    u64 first = 0, G = 0;
    for (u64 k = 0; k < a.K; k++) {
        std::unique_ptr<swg_paf> f(new swg_paf());
        std::string err;
        if (!paf_open_text(a.in[k], f.get(), &err)) {
            if (access(a.in[k], R_OK) == 0) throw RangeError{file_name(a, k) + ": " + err};
            throw IoError{file_name(a, k) + ": " + err};
        }
        const u64 b = f->text_len + (f->text_len && f->text[f->text_len - 1] != '\n' ? 1 : 0);
        // lines are estimated at 64 bytes or more (a PAF record has twelve fields); the newline scan checks the true count and
        // a union that needs more is split then (GroupTooLarge), before anything of it is written
        if (!group.empty() && !(group.size() < file_cap && G + b <= byte_cap && (G + b) / 64 < 0x7FFFFFF0ull &&
                                paf_union_memory(G + b, (G + b) / 64) <= mem_budget)) {
            filter_paf_group(a, first, group, mem_budget, S);
            group.clear();
            G = 0;
        }
        if (group.empty()) first = k;
        G += b;
        group.push_back(std::move(f));
    }
    if (!group.empty()) filter_paf_group(a, first, group, mem_budget, S);
    if (a.stats) *a.stats = S;
}

} // namespace swg

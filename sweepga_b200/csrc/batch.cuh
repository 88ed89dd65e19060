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
__device__ __forceinline__ u32 batch_table_of(const u32 *off, u32 K, u32 i) {
    u32 lo = 0, hi = K;
    while (hi - lo > 1) {
        const u32 mid = (lo + hi) >> 1;
        if (off[mid] <= i) lo = mid;
        else hi = mid;
    }
    return lo;
}
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

} // namespace swg

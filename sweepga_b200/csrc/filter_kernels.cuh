// filter_kernels.cuh — the sm_100a kernels of the mapping filter.
//
// Each kernel cites the reference code it replaces (paths relative to /root/reference).
// All parity-critical f64 expressions use explicit round-to-nearest intrinsics or are plain
// IEEE ops compiled with -fmad=false (no contraction).  No tensor cores: nothing here is a
// dense contraction; every kernel is HBM/L2 bound integer/byte work.
#pragma once
#include "common.cuh"
#include "scan.cuh"
#include "group_sort.cuh"
#include "glibc_log.cuh"

namespace swg {

// flags[i] bits
constexpr u8 F_ALIVE = 1;   // passed the stage-1 retain (paf_filter.rs:384-388)
constexpr u8 F_ZLQ = 2;     // zero-length query interval
constexpr u8 F_ZLT = 4;     // zero-length target interval
constexpr u8 F_PREMEM = 8;  // member of a chain that passed the mass/identity filter (pre_sweep_scaffold_members)
constexpr u8 F_REV = 16;    // reverse strand (any strand byte other than '+', paf_filter.rs:311)
constexpr u8 F_ANCHOR = 32; // status == scaffold: member of a kept chain or captured inversion (set by k_assign / t_inversion)

// counters (u64 each) shared with the host
enum {
    C_ALIVE = 0, C_ZLQ, C_ZLT, C_MAXCOORD, C_BAD, C_KEPT_M, C_GROUPS, C_CHAINS, C_PASS, C_PASS_ZEROSPAN,
    C_KEPT_CHAINS, C_ANCHORS, C_RESCUED, C_KEPT, C_NEAR_TIES, C_WORK, C_INV, C_HUGE, C_TMP0, C_RUNS, C_COUNT = 32
};

struct DevIn {
    const u32 *qid, *tid, *qs, *qe, *ts, *te, *blen, *matches;
    const double *identity;
    const u8 *strand;
    const double *score; // optional
    const u32 *P, *P2;
    u32 n, n_seq;
};

// ---------------------------------------------------------------------------------------------
// open-addressing hash: genome pair (P(q),P(t)) -> min record index ("first appearance" of the
// IndexMap at paf_filter.rs:1037-1046)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ u32 hash64(u64 k) {
    k ^= k >> 33; k *= 0xff51afd7ed558ccdULL; k ^= k >> 33; k *= 0xc4ceb9fe1a85ec53ULL; k ^= k >> 33;
    return (u32)k;
}
__device__ __forceinline__ void hash_insert_min(u64 *hk, u32 *hv, u32 mask, u64 key, u32 val) {
    u32 s = hash64(key) & mask;
    while (true) {
        u64 prev = atomicCAS((unsigned long long *)&hk[s], (unsigned long long)NONE64, (unsigned long long)key);
        if (prev == NONE64 || prev == key) { atomicMin(&hv[s], val); return; }
        s = (s + 1) & mask;
    }
}
__device__ __forceinline__ u32 hash_lookup(const u64 *hk, const u32 *hv, u32 mask, u64 key) {
    u32 s = hash64(key) & mask;
    while (true) {
        u64 k = hk[s];
        if (k == key) return hv[s];
        if (k == NONE64) return NONE32;
        s = (s + 1) & mask;
    }
}


// add per-thread small counts into a u64 counter: warp reduce, then one atomic per CTA
// (same-address global atomics cost ~0.5 ns each; one per warp was the top cost of the flat kernels)
template <int NC> __device__ __forceinline__ void block_count_add(u64 *ctr, const int (&slot)[NC], const u32 (&val)[NC]) {
    __shared__ u32 s_part[NC];
    if (threadIdx.x < NC) s_part[threadIdx.x] = 0;
    __syncthreads();
#pragma unroll
    for (int k = 0; k < NC; k++) {
        u32 w = __reduce_add_sync(0xFFFFFFFFu, val[k]);
        if (lane_id() == 0 && w) atomicAdd(&s_part[k], w);
    }
    __syncthreads();
    if (threadIdx.x < NC && s_part[threadIdx.x]) atomicAdd((unsigned long long *)&ctr[slot[threadIdx.x]], (unsigned long long)s_part[threadIdx.x]);
}

// ---------------------------------------------------------------------------------------------
// K0: stage-1 retain + range checks + genome-pair first appearance  (paf_filter.rs:384-388)
// 33 B read + 1 B written per record.
// ---------------------------------------------------------------------------------------------
// identity column, or (identity == NULL) the parser's default matches / max(block_length, 1) (paf_filter.rs:322): one IEEE
// division of two exactly converted integers, the same bits as the host's
__device__ __forceinline__ double rec_identity(const DevIn &in, u32 i) {
    if (in.identity) return in.identity[i];
    const u32 b = in.blen[i];
    return __ddiv_rn((double)in.matches[i], (double)(b > 1 ? b : 1));
}

// KEYS: also writes the chain sort key of every record in the "gap layout" ((query, target, strand) << 32 | query_start) —
// the width of the coordinate field is only known after this kernel (rs_squeeze closes the gap inside the sort) — and the
// payload (the record index): the key pass of k_chain_keys without a second read of the columns.  Valid when the primary
// sweep is the closed form and no alive record has an empty interval (kept == alive); the host falls back to k_chain_keys
// otherwise.
template <bool KEYS>
__global__ void __launch_bounds__(256) k_prefilter(DevIn in, u64 min_len, double min_id, int keep_self, u8 *__restrict__ flags,
                                                   u64 *__restrict__ ctr, u64 *hk, u32 *hv, u32 hmask,
                                                   uint4 *__restrict__ rec4, int sb = 0, u64 *__restrict__ keys = nullptr,
                                                   u32 *__restrict__ vals = nullptr) {
    u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    bool alive = false, zq = false, zt = false, bad = false;
    u32 maxc = 0;
    u64 g = NONE64;
    u32 qt = NONE32; // (query, target, strand) as one word, for the run count below (ids beyond 2^15 alias: it is only an estimate)
    if (i < in.n) {
        u32 q = in.qid[i], t = in.tid[i];
        u32 qs = in.qs[i], qe = in.qe[i], ts = in.ts[i], te = in.te[i];
        const bool bad_id = q >= in.n_seq || t >= in.n_seq;
        const bool bad_iv = qe < qs || te < ts; // the marshaller's mark for "does not fit the u32 SoA" as well (paf_io.cpp)
        // without an identity column and with a threshold <= 0 the test is always true (matches / block >= 0): `matches`
        // is then not read here and its upload overlaps this kernel and the sort
        const bool id_ok = (!in.identity && min_id <= 0.0) ? true : rec_identity(in, i) >= min_id;
        alive = !bad_id && (min_len == 0 || (u64)in.blen[i] >= min_len) && (keep_self || q != t) && id_ok; // (min_len 0: block_length not read)
        // an impossible interval is an error only if the record survives the retain: the reference (u64, no check) would
        // have dropped it here too (paf_filter.rs:384-388)
        bad = bad_id || (alive && bad_iv);
        if (bad) alive = false;
        zq = alive && qe == qs;
        zt = alive && te == ts;
        maxc = alive ? max(qe, te) : 0u;
        if (alive) g = ((u64)in.P[q] << 32) | in.P[t];
        const bool rev = in.strand[i] != '+';
        qt = (q << 17) ^ (t << 1) ^ (rev ? 1u : 0u);
        flags[i] = (u8)((alive ? F_ALIVE : 0) | (zq ? F_ZLQ : 0) | (zt ? F_ZLT : 0) | (rev ? F_REV : 0));
        if (KEYS) {
            const u64 grp = alive ? ((((u64)q << sb) | t) << 1 | (rev ? 1 : 0)) : ((1ull << (2 * sb + 1)) - 1); // dead: all ones, sorts last
            keys[i] = (grp << 32) | (alive ? qs : 0xFFFFFFFFu);
            vals[i] = i;
        }
        // packed copy for the post-sort gather: one 16 B sector instead of four 4 B gathers.  `matches` is NOT touched
        // here (unless identity has to be derived from it): it is first read by the gather after the sort, so its
        // host-to-device copy can overlap K0 + sort.
        if (rec4) rec4[i] = make_uint4(qs, qe, ts, te);
    }
    const u32 full = 0xFFFFFFFFu;
    // runs of consecutive records with one (query, target, strand): how grouped the input is (the record sort picks its method by
    // it).  Warp starts count as run starts: an over-estimate by at most n / 32.
    u32 prev_qt = __shfl_up_sync(full, qt, 1);
    const bool head = i < in.n && (lane_id() == 0 || prev_qt != qt);
    {
        const int slots[5] = {C_ALIVE, C_ZLQ, C_ZLT, C_BAD, C_RUNS};
        const u32 vals[5] = {alive ? 1u : 0u, zq ? 1u : 0u, zt ? 1u : 0u, bad ? 1u : 0u, head ? 1u : 0u};
        block_count_add<5>(ctr, slots, vals);
    }
    u32 mx = __reduce_max_sync(full, maxc);
    if (lane_id() == 0 && mx > (u32)ctr[C_MAXCOORD]) atomicMax((unsigned long long *)&ctr[C_MAXCOORD], (unsigned long long)mx);
    // one hash insert per distinct genome pair per warp; the lowest lane holds the lowest index.  Records of one
    // genome pair are normally contiguous, so the whole warp usually shares the pair: two votes instead of MATCH.ANY.
    const u32 alive_mask = __ballot_sync(full, alive);
    if (alive_mask == 0) return;
    const u32 first = __ffs(alive_mask) - 1;
    const u64 g0 = __shfl_sync(full, g, first);
    u32 leader_of_mine;
    if (__all_sync(full, !alive || g == g0)) leader_of_mine = first;
    else leader_of_mine = __ffs(__match_any_sync(full, g)) - 1;
    if (alive && lane_id() == leader_of_mine) {
        // values only decrease: a plain read that already shows a smaller index makes the atomics unnecessary
        u32 sl = hash64(g) & hmask;
        bool done = false;
        for (int probe = 0; probe < 4; probe++) {
            u64 k = hk[sl];
            if (k == g) { done = hv[sl] <= i; break; }
            if (k == NONE64) break;
            sl = (sl + 1) & hmask;
        }
        if (!done) hash_insert_min(hk, hv, hmask, g, i);
    }
}

// ---------------------------------------------------------------------------------------------
// K1: chain sort keys for the mappings that survived the primary sweep (the set M).
// key = (qid | tid | strand | query_start): replaces the (query,target,strand) IndexMap +
// stable sort_by_key(query_start) of paf_filter.rs:761-777.   keep_q/keep_t may be NULL
// (closed form: every alive mapping with a non-empty interval survives an n = inf sweep).
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_chain_keys(DevIn in, const u8 *__restrict__ flags, const u8 *__restrict__ keep_q,
                                                    const u8 *__restrict__ keep_t, int sb, int cb, u64 *__restrict__ keys,
                                                    u32 *__restrict__ vals, u64 *__restrict__ ctr) {
    u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    bool kept = false;
    if (i < in.n) {
        const u8 fl = flags[i];
        kept = (fl & F_ALIVE) && (!keep_q || keep_q[i]) && (!keep_t || keep_t[i]);
        // dead records: all ones in the key's own 2*sb + 1 + cb bits (ids stay below 2^sb - 1, so they sort behind every
        // live key) and zero above, so that the word still fits after the packed sort has shifted it
        const int kb = 2 * sb + 1 + cb;
        u64 k = kb >= 64 ? NONE64 : ((1ull << kb) - 1);
        if (kept) {
            u64 sbit = (fl & F_REV) ? 1 : 0;
            k = ((((u64)in.qid[i] << sb | in.tid[i]) << 1 | sbit) << cb) | in.qs[i];
        }
        keys[i] = k;
        vals[i] = i;
    }
    const int slots[1] = {C_KEPT_M};
    const u32 cvals[1] = {kept ? 1u : 0u};
    block_count_add<1>(ctr, slots, cvals);
}

// scaffold_gap == 0 exit (paf_filter.rs:409-434): survivors are Unassigned, no chain id
__global__ void __launch_bounds__(256) k_unassigned(u32 n, const u8 *__restrict__ flags, const u8 *__restrict__ keep_q,
                                                    const u8 *__restrict__ keep_t, u8 *__restrict__ status, u64 *__restrict__ ctr) {
    u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    bool kept = false;
    if (i < n) {
        kept = (flags[i] & F_ALIVE) && (!keep_q || keep_q[i]) && (!keep_t || keep_t[i]);
        status[i] = kept ? 3 : 0;
    }
    const int slots[1] = {C_KEPT};
    const u32 vals[1] = {kept ? 1u : 0u};
    block_count_add<1>(ctr, slots, vals);
}

// ---------------------------------------------------------------------------------------------
// K3: best-buddy chaining (paf_filter.rs:780-851), union-find roots (union_find.rs:25-41: the root of a
// set is always its head) and per-chain aggregates (paf_filter.rs:875-894), in three phases:
//   P1 k_chain_candidates  flat, one thread per position: the unconstrained best successor u(i)
//                          (smallest d, first minimal j) — all of the O(window) gap arithmetic, coalesced.
//   P2 k_chain_resolve     the inherently sequential part, one thread per group: walk i ascending;
//                          if u(i) still beats best_pred_score[u(i)] it IS the reference's choice (the global
//                          arg-min is eligible, so it is the arg-min over the eligible ones); only a blocked
//                          i re-scans its window with the eligibility test.  ~10 instructions per step.
//   P3 k_chain_heads / k_chain_members  flat: bounding boxes and sums per chain (segmented warp
//                          reduction, then one atomic set per run).
// ---------------------------------------------------------------------------------------------
// sorted position -> input index: the payload column of a pairs sort, or the low bits of the packed words
struct SortedIdx {
    const u64 *w;
    const u32 *v;
    u64 mask;
    __device__ __forceinline__ u32 operator[](u32 p) const { return w ? (u32)(w[p] & mask) : v[p]; }
};
struct Cand { // unconstrained best successor of a position
    u64 d;    // squared gap distance
    u32 j;    // sorted position of the successor, NONE32 if the window holds no valid candidate
    u32 c0;   // first position past the linear phase whose query_start >= query_end (NONE32 if the search never got there):
              // the origin of the outward scans, reused by the re-scans of the resolve
};

// gap rule of paf_filter.rs:799-833 (query axis and, strand-aware, target axis)
// 32-bit arithmetic up to the squares: coordinates are u32 and the host refuses scaffold_gap >= 2^31, so every gap and
// G + 1 fit (the reference computes the same values in u64).
__device__ __forceinline__ bool bb_candidate(const uint4 &a, const uint4 &b, bool fwd, u64 G, u64 G5, u64 &d) {
    const u32 g = (u32)G, g5 = (u32)G5;
    u32 qgap, rgap;
    if (b.x >= a.y) qgap = b.x - a.y;
    else { const u32 ov = a.y - b.x; qgap = ov <= g5 ? ov : g + 1; }
    if (fwd) {
        if (b.z >= a.w) rgap = b.z - a.w;
        else { const u32 ov = a.w - b.z; rgap = ov <= g5 ? ov : g + 1; }
    } else {
        if (a.z >= b.w) rgap = a.z - b.w;
        else { const u32 ov = b.w - a.z; rgap = ov <= g5 ? ov : g + 1; }
    }
    if (qgap <= g && rgap <= g) { d = (u64)qgap * qgap + (u64)rgap * rgap; return true; }
    return false;
}

// Arg-min over the successors of position i inside its group (.., e): smallest d, then smallest j ("first minimal
// j", paf_filter.rs:791-843); ELIG adds the reference's eligibility test d < best_pred_score[j].
// The first BB_LINEAR successors are scanned in order (ordinary data: a handful of candidates).  If the window goes
// on (dense piles: 10^4..10^5 candidates) the rest is searched outwards from the first position whose query_start
// reaches query_end(i): d >= q_gap^2 and q_gap grows monotonically in both directions from there, so the scan stops
// as soon as q_gap^2 exceeds the best d found — exact, and near-constant work per position in a dense pile.
constexpr u32 BB_LINEAR = 48;
template <bool ELIG>
__device__ __forceinline__ void bb_best_successor(const uint4 *__restrict__ srec, const u64 *bps, u32 i, u32 e, const uint4 &a,
                                                  bool fwd, u64 G, u64 G5, u64 &bd, u32 &bj, u32 *c0_out = nullptr, bool *linear_only = nullptr) {
    const u64 bound = (u64)a.y + G;
    bd = NONE64;
    bj = NONE32;
    if (c0_out) *c0_out = NONE32;
    u32 j = i + 1;
    const u32 lin_end = min(e, i + 1 + BB_LINEAR);
    for (; j < lin_end; j++) {
        const uint4 b = srec[j];
        if ((u64)b.x > bound) return; // window exhausted
        u64 d;
        if (bb_candidate(a, b, fwd, G, G5, d) && d < bd && (!ELIG || d < bps[j])) { bd = d; bj = j; }
    }
    if (j >= e) return;
    if (linear_only) { *linear_only = true; return; } // the window goes on past the linear phase and the caller does not want the rest
    u32 lo = j, hi = e; // first position in [j, e) with query_start >= query_end(i)
    while (lo < hi) {
        const u32 mid = (lo + hi) >> 1;
        if (srec[mid].x < a.y) lo = mid + 1; else hi = mid;
    }
    const u32 c0 = lo;
    if (c0_out) *c0_out = c0;
    for (u32 r = c0; r < e; r++) { // right: q_gap = qs - qe >= 0, non-decreasing
        const uint4 b = srec[r];
        const u64 qg = (u64)b.x - a.y;
        if (qg > G || qg * qg > bd) break;
        u64 d;
        if (bb_candidate(a, b, fwd, G, G5, d) && (d < bd || (d == bd && r < bj)) && (!ELIG || d < bps[r])) { bd = d; bj = r; }
    }
    for (u32 l = c0; l > j;) { // left: overlap = qe - qs > 0, non-decreasing going left
        l--;
        const uint4 b = srec[l];
        const u64 ov = (u64)a.y - b.x;
        if (ov > G5 || ov * ov > bd) break;
        u64 d;
        if (bb_candidate(a, b, fwd, G, G5, d) && (d < bd || (d == bd && l < bj)) && (!ELIG || d < bps[l])) { bd = d; bj = l; }
    }
}

// P1: 24 B read (+ window re-reads served by L1) and 16 B written per position, plus one 32-bit exchange per candidate:
// position p CLAIMS its unconstrained best successor, pred[j] = p.  If every successor of a group is claimed at most once,
// the reference's loop does exactly that: best_pred_score[j] is still "none" when its only picker arrives, so the picker's
// unconstrained arg-min is eligible and taken (paf_filter.rs:835-850).  A second claim on some j marks the whole group
// dirty; dirty groups (rare on ordinary data) are redone by the sequential resolve below, which rewrites their pred[].
// pred[] must be NONE32 everywhere on entry.
// LIST = false: one thread per position, claims only (the 16 B candidate record is not written: clean groups never read it).
// LIST = true: grid-stride over a list of positions (those of the dirty and huge groups), writes their candidate records
// for the resolve kernels / the fixed-point iteration; no claims.
constexpr u32 RES_SMALL = 16;
constexpr u32 RES_THREAD_MAX = 16; // dirty groups up to this size are walked by one thread (from registers), larger ones by a warp
// 8 CTAs per SM (32 registers): the window scan is a chain of dependent loads, hidden only by resident warps; the bound costs one
// 4 B spill of the loop index per position, outside the scan (40 registers without it: 268 against 220 us per 20 M positions)
template <bool LIST>
__global__ void __launch_bounds__(256, 8)
k_chain_candidates(const uint4 *__restrict__ srec, const u64 *__restrict__ skey, const u32 *__restrict__ gid,
                   const u32 *__restrict__ gstart, u32 n_groups, u32 n_m, int cb, u64 G, Cand *__restrict__ cand,
                   u32 *pred, u32 *grp_dirty, const u32 *__restrict__ list, const u32 *__restrict__ n_list_ptr, u32 fx_min = 0,
                   u32 *work = nullptr, u32 *work_big = nullptr, u32 *bb_ctr = nullptr) {
    const u32 n_items = LIST ? *n_list_ptr : n_m;
    for (u32 x = blockIdx.x * blockDim.x + threadIdx.x; x < n_items; x += gridDim.x * blockDim.x) {
        const u32 p = LIST ? list[x] : x;
        const uint4 a = srec[p]; // x=qs y=qe z=ts w=te
        const bool fwd = ((skey[p] >> cb) & 1) == 0;
        const u32 g = gid[p];
        const u32 e = (g + 1 < n_groups) ? gstart[g + 1] : n_m;
        if (!LIST && fx_min != NONE32 && e - gstart[g] >= fx_min) continue; // huge group: the fixed-point iteration searches itself
                                                                              // (the host passes NONE32 when no group is huge)
        u64 bd;
        u32 bj;
        u32 c0;
        bb_best_successor<false>(srec, nullptr, p, e, a, fwd, G, G / 5, bd, bj, &c0);
        if (LIST) {
            Cand c;
            c.d = bd; c.j = bj; c.c0 = c0;
            cand[p] = c;
        } else if (bj != NONE32 && atomicExch(&pred[bj], p) != NONE32 && atomicExch(&grp_dirty[g], 1u) == 0) {
            // first conflict seen in this group: it goes on a work list of the sequential resolve — the thread walk for small
            // groups, the warp walk for larger or dense ones (a thread pays one memory round trip per step; with only the dirty
            // groups listed, the longest walk is the kernel time).  Huge groups have their own path.  The order of a list does
            // not matter: every group is resolved on its own.
            const u32 s0 = gstart[g];
            const u64 size = e - s0;
            if (size < fx_min) {
                const u64 span = (u64)srec[e - 1].x - srec[s0].x + 1;
                const bool big = size > RES_THREAD_MAX || size * G > 64 * span;
                if (big) work_big[atomicAdd(&bb_ctr[2], 1u)] = g;
                else work[atomicAdd(&bb_ctr[0], 1u)] = g;
            }
        }
    }
}

// The candidate records of the positions of LISTED GROUPS (the dirty ones), one warp per group, lanes over its positions.
__global__ void __launch_bounds__(256)
k_chain_candidates_groups(const uint4 *__restrict__ srec, const u64 *__restrict__ skey, const u32 *__restrict__ gstart, u32 n_groups, u32 n_m, int cb,
                          u64 G, Cand *__restrict__ cand, const u32 *__restrict__ glist_a, const u32 *__restrict__ n_a, const u32 *__restrict__ glist_b,
                          const u32 *__restrict__ n_b) {
    const u32 na = *n_a, nb = *n_b;
    const u32 lane = lane_id();
    for (u32 w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < na + nb; w += (gridDim.x * blockDim.x) >> 5) {
        const u32 g = w < na ? glist_a[w] : glist_b[w - na];
        const u32 s0 = gstart[g], e = (g + 1 < n_groups) ? gstart[g + 1] : n_m;
        const bool fwd = ((skey[s0] >> cb) & 1) == 0;
        for (u32 p = s0 + lane; p < e; p += 32) {
            const uint4 a = srec[p];
            Cand c;
            bb_best_successor<false>(srec, nullptr, p, e, a, fwd, G, G / 5, c.d, c.j, &c.c0);
            cand[p] = c;
        }
    }
}

// P2: the reference's sequential loop for the DIRTY groups (some successor claimed twice), one thread per group; lanes
// refill from the work list as they finish.  The whole state of a group is local to it (candidates point inside the
// group), so the thread first resets the group's best_pred_score / pred and then walks it; a step is "does the
// unconstrained arg-min still beat best_pred_score?" (then it is the reference's pick: the global arg-min is eligible, so
// it is the arg-min over the eligible ones); only a blocked step re-scans its window with the eligibility test.
// Result: pred[j] = best_pred_idx[j] (paf_filter.rs:847-850), NONE32 = no predecessor.
__global__ void __launch_bounds__(128)
k_chain_resolve(const Cand *__restrict__ cand, const uint4 *__restrict__ srec, const u64 *__restrict__ skey,
                const u32 *__restrict__ gstart, u32 n_groups, u32 n_m, const u32 *__restrict__ work, const u32 *__restrict__ n_work_ptr,
                int cb, u64 G, u64 *bps, u32 *pred, u32 *work_counter) {
    const u32 full = 0xFFFFFFFFu;
    const u64 G5 = G / 5;
    const u32 n_work = *n_work_ptr;
    bool active = false, exhausted = false, fwd = true;
    u32 e = 0, i = 0;
    Cand c_cur{0, NONE32, 0}, c_next{0, NONE32, 0};
    u64 b_cur = 0;
    while (true) {
        const u32 need = __ballot_sync(full, !active && !exhausted);
        if (need) {
            const u32 leader = __ffs(need) - 1;
            u32 base = 0;
            if (lane_id() == leader) base = atomicAdd(work_counter, (u32)__popc(need));
            base = __shfl_sync(full, base, leader);
            if (!active && !exhausted) {
                const u32 w = base + __popc(need & lanemask_lt());
                if (w >= n_work) exhausted = true;
                else {
                    const u32 g = work[w];
                    i = gstart[g];
                    e = (g + 1 < n_groups) ? gstart[g + 1] : n_m;
                    fwd = ((skey[i] >> cb) & 1) == 0;
                    active = true;
                    const u32 n = e - i;
                    if (n <= RES_SMALL) {
                        // a small group is resolved from ONE burst of loads (its candidates) on per-thread copies
                        Cand cs[RES_SMALL];
                        u32 pr[RES_SMALL];
                        u64 bp[RES_SMALL];
#pragma unroll
                        for (u32 k = 0; k < RES_SMALL; k++) {
                            if (k < n) cs[k] = cand[i + k];
                            pr[k] = NONE32;
                            bp[k] = NONE64;
                        }
                        u32 k = 0;
                        bool blocked = false;
                        for (; k + 1 < n; k++) {
                            const Cand c = cs[k];
                            if (c.j == NONE32) continue;
                            const u32 jj = c.j - i;
                            if (c.d < bp[jj]) { bp[jj] = c.d; pr[jj] = i + k; }
                            else { blocked = true; break; } // needs the arg-min over the eligible candidates: generic walk
                        }
                        for (u32 q = 0; q < n; q++) pred[i + q] = pr[q];
                        if (!blocked) {
                            active = false;
                        } else { // publish the state reached so far; the generic walk continues at step k
                            for (u32 q = 0; q < n; q++) bps[i + q] = bp[q];
                            c_cur = cs[k];
                            c_next = (k + 1 < n) ? cs[k + 1] : Cand{0, NONE32, 0};
                            b_cur = bp[c_cur.j - i];
                            i += k;
                        }
                    } else {
                        for (u32 q = i; q < e; q++) { bps[q] = NONE64; pred[q] = NONE32; }
                        c_cur = cand[i];
                        c_next = (i + 1 < e) ? cand[i + 1] : Cand{0, NONE32, 0};
                        b_cur = NONE64;
                    }
                }
            }
        }
        if (__all_sync(full, exhausted && !active)) break;
        if (active) {
            // software pipeline: the loads of step i+1 (its candidate, that candidate's best_pred_score) are issued before
            // step i is decided; step i's own store is forwarded in registers.
            const Cand c_nn = (i + 2 < e) ? cand[i + 2] : Cand{0, NONE32, 0}; // two steps ahead: its address is free
            u64 b_next = (c_next.j != NONE32) ? bps[c_next.j] : 0;             // c_next was loaded one step ago
            u32 chosen = NONE32;
            u64 chosen_d = 0;
            if (c_cur.j != NONE32) {
                if (c_cur.d < b_cur) { // the unconstrained arg-min is eligible => it is the reference's pick
                    chosen = c_cur.j;
                    chosen_d = c_cur.d;
                } else { // blocked: arg-min over the eligible candidates (paf_filter.rs:835-843)
                    const uint4 a = srec[i];
                    u64 bd;
                    u32 bj;
                    bb_best_successor<true>(srec, bps, i, e, a, fwd, G, G5, bd, bj);
                    chosen = bj;
                    chosen_d = bd;
                }
                if (chosen != NONE32) {
                    bps[chosen] = chosen_d;
                    pred[chosen] = i;
                    if (chosen == c_next.j) b_next = chosen_d; // supersedes the value prefetched above
                }
            }
            c_cur = c_next;
            c_next = c_nn;
            b_cur = b_next;
            if (++i == e) active = false;
        }
    }
}

// P2b: the same resolve for LARGE or DENSE groups, one warp per group.  The step is decided by the whole warp; a
// blocked step searches its window with 32 lanes (coalesced chunks), with the same q_gap^2 pruning as
// bb_best_successor: a single thread would pay one dependent-load latency per candidate.
__device__ __forceinline__ void bb_argmin(u64 &bd, u32 &bj) { // smallest d, then smallest j
    const u32 full = 0xFFFFFFFFu;
    u32 hi = (u32)(bd >> 32), lo = (u32)bd;
    u32 mh = __reduce_min_sync(full, hi);
    u32 ml = __reduce_min_sync(full, hi == mh ? lo : 0xFFFFFFFFu);
    bool is = hi == mh && lo == ml;
    bj = __reduce_min_sync(full, is ? bj : NONE32);
    bd = ((u64)mh << 32) | ml;
}
#ifndef SWG_RESCAN_WIDTH
#define SWG_RESCAN_WIDTH 128
#endif
// The blocked step of the sequential walk: the arg-min over the candidates j that pass the eligibility test d < bps[j].
__device__ __forceinline__ void bb_best_successor_warp(const uint4 *__restrict__ srec, const u64 *bps, u32 i, u32 e, const uint4 &a,
                                                       bool fwd, u64 G, u64 G5, u64 &bd, u32 &bj, u32 c0_hint) {
    const u32 full = 0xFFFFFFFFu;
    const u32 lane = lane_id();
    const u64 bound = (u64)a.y + G;
    constexpr u32 RW = SWG_RESCAN_WIDTH; // candidates per outward round: four 32-wide chunks, loads independent, one warp arg-min
    bd = NONE64;
    bj = NONE32;
    const u32 lin_end = min(e, i + 1 + 64);
    const u32 jl = lin_end; // the outward scans cover [jl, e)
    u32 rbase, ltop;        // where the outward rounds continue
    u64 rnext = NONE64, lnext = NONE64; // query_start of the first candidate of the next right / left round (NONE64: none)
    if (c0_hint != NONE32 && lin_end < e) {
        // The origin of the outward scans is known from the candidate pass (its linear phase is shorter: hence the max).
        // First round: the 64 nearest successors, RW candidates to the right of the origin and RW to its left, all loads
        // in flight together — one L2 round trip and one arg-min instead of three of each.  Every candidate is validated
        // on its own (inside the window; gap rule), so evaluating this superset gives the same arg-min.
        const u32 c0 = max(c0_hint, jl);
        u64 ld = NONE64;
        u32 lj = NONE32;
        const u32 lcnt = min(RW, c0 - jl);
        // every load of the round is issued before the first use (bps too: its address does not depend on the record)
        uint4 rb[2 + 2 * (RW / 32)];
        u64 rp[2 + 2 * (RW / 32)];
        u32 rj[2 + 2 * (RW / 32)];
#pragma unroll
        for (u32 k = 0; k < 2; k++) {
            const u32 j = i + 1 + k * 32 + lane;
            rj[k] = j < lin_end ? j : NONE32;
        }
#pragma unroll
        for (u32 k = 0; k < RW / 32; k++) {
            const u32 r = c0 + k * 32 + lane;
            rj[2 + k] = r < e ? r : NONE32;
            const u32 off = k * 32 + lane;
            rj[2 + RW / 32 + k] = off < lcnt ? c0 - 1 - off : NONE32;
        }
#pragma unroll
        for (u32 k = 0; k < 2 + 2 * (RW / 32); k++)
            if (rj[k] != NONE32) { rb[k] = srec[rj[k]]; rp[k] = bps[rj[k]]; }
        rnext = c0 + RW < e ? (u64)srec[c0 + RW].x : NONE64; // first candidate of the next right round (pruning test)
        lnext = c0 - lcnt > jl ? (u64)srec[c0 - lcnt - 1].x : NONE64;
#pragma unroll
        for (u32 k = 0; k < 2 + 2 * (RW / 32); k++) {
            if (rj[k] == NONE32) continue;
            const uint4 b = rb[k];
            bool inwin;
            if (k < 2) inwin = (u64)b.x <= bound;                       // nearest successors: inside the window
            else if (k < 2 + RW / 32) inwin = (u64)b.x - a.y <= G;      // right of the origin: q_gap <= G
            else inwin = true;                                          // left of the origin: overlap, judged by the gap rule
            u64 d;
            if (inwin && bb_candidate(a, b, fwd, G, G5, d) && (d < ld || (d == ld && rj[k] < lj)) && d < rp[k]) { ld = d; lj = rj[k]; }
        }
        bb_argmin(ld, lj);
        bd = ld;
        bj = lj;
        rbase = c0 + RW;
        ltop = c0 - lcnt;
    } else {
        // linear phase: the first 64 successors (two chunks)
        u32 j0 = i + 1;
        bool exhausted = false;
        for (; j0 < lin_end && !exhausted; j0 += 32) {
            const u32 j = j0 + lane;
            bool inwin = false;
            if (j < lin_end) {
                const uint4 b = srec[j];
                inwin = (u64)b.x <= bound;
                u64 d;
                if (inwin && bb_candidate(a, b, fwd, G, G5, d) && (d < bd || (d == bd && j < bj)) && d < bps[j]) { bd = d; bj = j; }
            }
            exhausted = !__all_sync(full, inwin || j >= lin_end);
        }
        bb_argmin(bd, bj);
        if (exhausted || lin_end >= e) return;
        // first position in [jl, e) whose start is >= query_end: 33-ary search, 32 probes in flight per round (a binary
        // search pays one L2 round trip per halving: ~19 dependent loads in a 500 k-mapping group)
        u32 lo = jl, hi = e;
        while (hi - lo > 32) {
            const u32 width = hi - lo;
            const u32 p = lo + (u32)(((u64)(lane + 1) * width) / 33);
            const u32 below = __popc(__ballot_sync(full, srec[p].x < a.y)); // monotone: the first `below` probes are < query_end
            const u32 nlo = below ? lo + (u32)(((u64)below * width) / 33) + 1 : lo;
            const u32 nhi = below < 32 ? lo + (u32)(((u64)(below + 1) * width) / 33) : hi;
            lo = nlo;
            hi = nhi;
        }
        if (hi > lo) {
            const u32 p = lo + lane;
            const u32 below = __popc(__ballot_sync(full, p < hi && srec[p].x < a.y));
            lo += below;
        }
        rbase = lo;
        ltop = lo;
        rnext = rbase < e ? (u64)srec[rbase].x : NONE64;
        lnext = ltop > jl ? (u64)srec[ltop - 1].x : NONE64;
    }
    // Outward rounds.  The pruning test looks at the first candidate of a round only; candidates past the exact pruning
    // point have d >= q_gap^2 > best d and cannot win, so reading a few more of them changes nothing.
    for (u32 base = rbase; base < e; base += RW) { // right side, q_gap >= 0 non-decreasing
        const u64 qg0 = rnext - a.y;
        if (rnext == NONE64 || qg0 > G || qg0 * qg0 > bd) break;
        uint4 rb[RW / 32];
        u64 rp[RW / 32];
#pragma unroll
        for (u32 k = 0; k < RW / 32; k++) {
            const u32 r = base + k * 32 + lane;
            if (r < e) { rb[k] = srec[r]; rp[k] = bps[r]; }
        }
        rnext = base + RW < e ? (u64)srec[base + RW].x : NONE64;
        u64 ld = bd; // every lane starts from the best so far: only a candidate that beats it is tested for eligibility
        u32 lj = bj;
#pragma unroll
        for (u32 k = 0; k < RW / 32; k++) {
            const u32 r = base + k * 32 + lane;
            if (r < e) {
                const u64 qg = (u64)rb[k].x - a.y;
                u64 d;
                if (qg <= G && bb_candidate(a, rb[k], fwd, G, G5, d) && d < ld && d < rp[k]) { ld = d; lj = r; } // r ascends: ties keep the smaller j
            }
        }
        bb_argmin(ld, lj);
        bd = ld;
        bj = lj;
    }
    for (u32 top = ltop; top > jl;) { // left side, overlap > 0 non-decreasing going left; round = [top-RW, top)
        const u64 ov0 = (u64)a.y - lnext;
        if (lnext == NONE64 || ov0 > G5 || ov0 * ov0 > bd) break;
        const u32 cnt = min(RW, top - jl);
        uint4 rb[RW / 32];
        u64 rp[RW / 32];
#pragma unroll
        for (u32 k = 0; k < RW / 32; k++) {
            const u32 off = k * 32 + lane;
            if (off < cnt) { rb[k] = srec[top - 1 - off]; rp[k] = bps[top - 1 - off]; }
        }
        lnext = top - cnt > jl ? (u64)srec[top - cnt - 1].x : NONE64;
        u64 ld = bd;
        u32 lj = bj;
#pragma unroll
        for (u32 k = 0; k < RW / 32; k++) {
            const u32 off = k * 32 + lane;
            if (off < cnt) {
                const u32 l = top - 1 - off;
                u64 d;
                if (bb_candidate(a, rb[k], fwd, G, G5, d) && (d < ld || (d == ld && l < lj)) && d < rp[k]) { ld = d; lj = l; }
            }
        }
        bb_argmin(ld, lj);
        bd = ld;
        bj = lj;
        top -= cnt;
    }
}
__global__ void __launch_bounds__(128)
k_chain_resolve_warp(const Cand *__restrict__ cand, const uint4 *__restrict__ srec, const u64 *__restrict__ skey,
                     const u32 *__restrict__ gstart, u32 n_groups, u32 n_m, const u32 *__restrict__ work, const u32 *__restrict__ n_work_ptr,
                     int cb, u64 G, u64 *bps, u32 *pred, u32 *work_counter) {
    const u32 full = 0xFFFFFFFFu;
    const u32 lane = lane_id();
    const u64 G5 = G / 5;
    const u32 n_work = *n_work_ptr;
    while (true) {
        u32 w = 0;
        if (lane == 0) w = atomicAdd(work_counter, 1u);
        w = __shfl_sync(full, w, 0);
        if (w >= n_work) break;
        const u32 g = work[w];
        const u32 s = gstart[g], e = (g + 1 < n_groups) ? gstart[g + 1] : n_m;
        const bool fwd = ((skey[s] >> cb) & 1) == 0;
        for (u32 q = s + lane; q < e; q += 32) { bps[q] = NONE64; pred[q] = NONE32; } // the group's state starts empty
        __syncwarp();
        // 32 steps per batch: lane k prefetches the candidate and the current best_pred_score of step base + k in one
        // round trip; the steps then run in order from registers.  A step that writes bps[j] patches the prefetched
        // copies of the later steps of the batch, so every step sees exactly the state the sequential walk would.
        for (u32 base = s; base + 1 < e; base += 32) {
            const u32 ik = base + lane;
            Cand ck;
            ck.d = 0; ck.j = NONE32; ck.c0 = NONE32;
            u64 bk = 0;
            if (ik + 1 < e) {
                ck = cand[ik];
                if (ck.j != NONE32) bk = bps[ck.j];
            }
            const u32 steps = min(32u, e - 1 - base);
            for (u32 t = 0; t < steps; t++) {
                const u32 cj = __shfl_sync(full, ck.j, t);
                if (cj == NONE32) continue;
                const u64 cd = __shfl_sync(full, ck.d, t);
                const u64 bt = __shfl_sync(full, bk, t);
                u64 wd = NONE64; // what this step writes: bps[wj] = wd, pred[wj] = i
                u32 wj = NONE32;
                const u32 i = base + t;
                if (cd < bt) { wd = cd; wj = cj; }
                else {
                    const uint4 a = srec[i];
                    bb_best_successor_warp(srec, bps, i, e, a, fwd, G, G5, wd, wj, __shfl_sync(full, ck.c0, t));
                }
                if (wj != NONE32) {
                    if (lane == 0) { bps[wj] = wd; pred[wj] = i; }
                    if (ck.j == wj) bk = wd;               // later steps of the batch that look at the same successor
                    __syncwarp();
                }
            }
        }
    }
}

// rough count of candidate evaluations the chaining will need (guards against an input that would run for hours)
// Also counts the positions that belong to huge groups (size >= fx_min): those are chained by the fixed-point iteration
// of chain_fixpoint.cuh instead of a sequential walk.
constexpr u32 FX_MIN_GROUP = 16384;
// ESTIMATE = false: only the huge-group count (two coalesced reads per group); the work estimate needs two gathers per group
// and is computed only when SWG_MAX_PAIR_EVALS asks for it.
template <bool ESTIMATE>
__global__ void __launch_bounds__(256)
k_chain_work_estimate(const uint4 *__restrict__ rec4, SortedIdx sidx, const u32 *__restrict__ gstart, const u32 *__restrict__ n_groups_ptr, u32 n_m,
                      u64 G, u32 fx_min, u64 *ctr) {
    const u32 n_groups = *n_groups_ptr; // grid-stride: the host has not read the group count yet
    u64 est = 0;
    for (u32 g = blockIdx.x * blockDim.x + threadIdx.x; g < n_groups; g += gridDim.x * blockDim.x) {
        const u32 s = gstart[g], e = (g + 1 < n_groups) ? gstart[g + 1] : n_m;
        const u64 size = e - s;
        if (size >= fx_min) atomicAdd((unsigned long long *)&ctr[C_HUGE], (unsigned long long)size); // a handful of groups at most
        if (ESTIMATE && size > 1) {
            const u64 span = (u64)rec4[sidx[e - 1]].x - rec4[sidx[s]].x + 1; // (runs before the gather: two reads per group)
            u64 win = size * G / span + 1; // expected candidates per step
            if (win > size) win = size;
            est += size * win;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) est += __shfl_down_sync(0xFFFFFFFFu, est, o);
    if (lane_id() == 0 && est) atomicAdd((unsigned long long *)&ctr[C_WORK], (unsigned long long)est);
}

// P2c: union-find roots and dense chain numbers in ONE pass over pred[] (union_find.rs:25-41: every union hangs the
// singleton j under find(pred[j]), so the root of a set is its head and pred[] is a forest of paths with pred[j] < j;
// chains are numbered by ascending head position, union_find.rs:52-63).
// A CTA takes a tile of 2048 consecutive sorted positions (tile ids in scheduling order); heads are numbered by a decoupled
// look-back over the tiles' head counts.  Every position is resolved to a head inside the tile or to an ancestor in an
// EARLIER tile without block-wide rounds: each warp owns 256 consecutive positions and walks them as 8 chunks of 32 in
// order; an ancestor inside the current chunk is followed by pointer jumping in registers (5 shuffle rounds cover 32 hops),
// one in an earlier chunk of the warp is read once from the warp's resolved slice in shared memory.  After one barrier, a
// position pointing into an earlier warp's range hops over those slices (at most 7 hops, each to an earlier warp).
// A position whose ancestor a lies in an earlier tile gets chain_of[p] = 0x80000000 | a (positions are < 2^31) instead of
// waiting for that tile: k_chain_aggregate, which runs after this kernel, follows such marks to a number and writes it back.
// Every chain_of[] entry is written.  PRESET: root[] already holds the final root of some positions (huge groups chained by
// the fixed-point iteration), NONE32 elsewhere.
struct ChainDense { // per-chain aggregates, rows indexed by chain number
    u32 *qmin, *qmax, *tmin, *tmax; // = ChainTable qs / qe / ts / te
    u64 *sum_matches, *sum_block;
    u32 *k;                         // chain_N of the chain (0 = not kept): cleared with the row
};
constexpr int CR_THREADS = 256, CR_ITEMS = 8, CR_TILE = CR_THREADS * CR_ITEMS;
static_assert(CR_THREADS == SC_THREADS, "k_chain_number uses the 256-thread block scan of scan.cuh");
// 8 CTAs per SM (32 registers): a tile is a short chain of latencies (tile id, loads, scan, look-back), so resident tiles are
// what hides them; 20 B of spills in the row-clearing loop, once per CTA (48 registers without the bound: 145 against 117 us)
template <bool PRESET>
__global__ void __launch_bounds__(CR_THREADS, 8)
k_chain_number(const u32 *__restrict__ pred, const u32 *__restrict__ root_preset, u32 n_m, u32 *__restrict__ chain_of, u32 *__restrict__ head_pos,
               u64 *status, u32 *tile_counter, u32 *n_chains_out, ChainDense cd) {
    __shared__ u32 anc[CR_TILE];
    __shared__ u32 ws[CR_THREADS / 32];
    __shared__ u32 s_tile, s_excl;
    const u32 full = 0xFFFFFFFFu;
    const u32 tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) s_tile = atomicAdd(tile_counter, 1u);
    __syncthreads();
    const u32 tile = s_tile;
    const u32 base = tile * CR_TILE;
    const u32 wl = warp * (32 * CR_ITEMS); // the warp's range [wl, wl + 256) of the tile; chunk k = [wl + 32 k, wl + 32 k + 32)
    // load (chunk k of the warp at lane: coalesced), ancestor = predecessor, preset root or the position itself (a head)
    u32 a[CR_ITEMS], hcnt = 0; // hcnt: heads of the warp's range
#pragma unroll
    for (int k = 0; k < CR_ITEMS; k++) {
        const u32 p = base + wl + 32 * k + lane;
        a[k] = p;
        if (p < n_m) {
            const u32 pr = pred[p];
            if (pr != NONE32) a[k] = pr;
            if (PRESET) { const u32 r = root_preset[p]; if (r != NONE32) a[k] = r; }
        }
        hcnt += __popc(__ballot_sync(full, p < n_m && a[k] == p));
    }
    // resolve inside the warp's range, chunk by chunk: afterwards a[k] is a head of the range or an ancestor before it
#pragma unroll
    for (int k = 0; k < CR_ITEMS; k++) {
        const u32 c0 = base + wl + 32 * k;
        u32 x = a[k];
#pragma unroll
        for (int r = 0; r < 5; r++) { // pred < position: a chunk holds at most 31 hops
            const bool in = x >= c0 && x < c0 + 32;
            const u32 y = __shfl_sync(full, x, in ? x - c0 : lane);
            if (in) x = y;
        }
        if (x >= base + wl && x < c0) x = anc[x - base]; // an earlier chunk of this warp: already resolved
        a[k] = x;
        anc[wl + 32 * k + lane] = x;
        __syncwarp();
    }
    // heads of the tile in position order: lane 0 of each warp enters the warp's head count, so its exclusive prefix is the
    // number of heads before the warp's range
    u32 tot;
    const u32 ex_local = block_exclusive_scan_256(lane == 0 ? hcnt : 0u, ws, tot); // its barriers also publish every warp's slice of anc[]
    if (tid < 32) {
        if (lane == 0) st_relaxed_u64(&status[tile], (tile == 0 ? SC_FLAG_INCL : SC_FLAG_AGG) | tot);
        u32 excl = 0;
        if (tile != 0) {
            i64 t = (i64)tile - 1;
            while (true) {
                const i64 mine = t - lane;
                const u64 w = mine >= 0 ? ld_relaxed_u64(&status[mine]) : SC_FLAG_INCL;
                const u32 incl = __ballot_sync(0xFFFFFFFFu, (w & SC_FLAG_INCL) != 0);
                const u32 ready = __ballot_sync(0xFFFFFFFFu, (w & (SC_FLAG_INCL | SC_FLAG_AGG)) != 0);
                const u32 upto = incl ? (u32)(__ffs(incl) - 1) : 31u;
                const u32 need = upto == 31 ? 0xFFFFFFFFu : ((2u << upto) - 1);
                if ((ready & need) != need) continue;
                excl += __reduce_add_sync(0xFFFFFFFFu, lane <= upto ? (u32)(w & SC_VAL_MASK) : 0u);
                if (incl) break;
                t -= 32;
            }
            if (lane == 0) st_relaxed_u64(&status[tile], SC_FLAG_INCL | (u64)(excl + tot));
        }
        if (lane == 0) {
            s_excl = excl;
            if ((u64)(tile + 1) * CR_TILE >= n_m) *n_chains_out = excl + tot;
        }
    }
    // an ancestor in an earlier warp's range: hop over the resolved slices (each hop lands on a head or goes to an earlier
    // warp) until a head of the tile or a position before the tile
#pragma unroll
    for (int k = 0; k < CR_ITEMS; k++) {
        u32 x = a[k];
        while (x >= base && x < base + wl) {
            const u32 y = anc[x - base];
            if (y == x) break;
            x = y;
        }
        a[k] = x;
    }
    __syncthreads(); // every read of the resolved slices is done, and s_excl is visible
    // heads get their numbers, in position order
    {
        u32 ex = s_excl + __shfl_sync(full, ex_local, 0); // heads of the tile before this warp's range
#pragma unroll
        for (int k = 0; k < CR_ITEMS; k++) {
            const u32 p = base + wl + 32 * k + lane;
            const u32 hmask = __ballot_sync(full, p < n_m && a[k] == p); // a head resolves to itself, nothing else does
            if ((hmask >> lane) & 1u) {
                const u32 r = ex + __popc(hmask & lanemask_lt());
                head_pos[r] = p;
                anc[wl + 32 * k + lane] = 0x80000000u | r; // marks "this entry now holds a chain number" (positions are < 2^31)
            }
            ex += __popc(hmask);
        }
    }
    // the tile's chains are the consecutive rows s_excl .. s_excl + tot of the aggregate table: they start empty (the host does
    // not know the chain count yet, so nobody else can clear them)
    for (u32 r = s_excl + tid, r_end = s_excl + tot; r < r_end; r += CR_THREADS) {
        cd.qmin[r] = NONE32; cd.qmax[r] = 0; cd.tmin[r] = NONE32; cd.tmax[r] = 0;
        cd.sum_matches[r] = 0; cd.sum_block[r] = 0; cd.k[r] = 0;
    }
    __syncthreads();
    // every position: chain number of its head (inside the tile) or the mark of its ancestor in an earlier tile
#pragma unroll
    for (int k = 0; k < CR_ITEMS; k++) {
        const u32 p = base + wl + 32 * k + lane;
        if (p >= n_m) continue;
        const u32 x = a[k];
        chain_of[p] = x >= base ? anc[x - base] & 0x7FFFFFFFu : 0x80000000u | x;
    }
}

// P3: per-chain aggregates (paf_filter.rs:875-894) into the dense chain table: bounding box by atomicMin / atomicMax, sums
// by atomicAdd; runs of one chain inside a warp are reduced first (one set of atomics per run).  Every position also feeds
// its group's min original index (the first appearance of the group in the input).  The table rows are pre-set to
// (max, 0, max, 0, 0, 0).
// A marked chain_of[p] (0x80000000 | ancestor, left by k_chain_number) is followed to a number, which is written back for
// k_assign.  Marks only ever point backwards and are only ever replaced by their number, so a racing reader sees the mark
// or the number: both lead to the same chain, in at most as many hops as the chain spans tiles.
__global__ void __launch_bounds__(256)
k_chain_aggregate(const uint4 *__restrict__ srec, const u32 *__restrict__ blen, const u32 *__restrict__ matches, SortedIdx sidx,
                  const u32 *__restrict__ gid, u32 *chain_of, u32 n_m, ChainDense cd, u32 *__restrict__ grp_minidx) {
    const u32 full = 0xFFFFFFFFu;
    const u32 lane = lane_id();
    const u32 p = blockIdx.x * blockDim.x + threadIdx.x;
    const bool ok = p < n_m;
    u32 g = NONE32, idx = NONE32, ci = 0x80000000u | lane; // lanes past the end never match anything
    uint4 a = make_uint4(NONE32, 0, NONE32, 0);
    uint2 m = make_uint2(0, 0);
    if (ok) {
        g = gid[p];
        idx = sidx[p];
        ci = chain_of[p];
        if (ci & 0x80000000u) {
            do { ci = chain_of[ci & 0x7FFFFFFFu]; } while (ci & 0x80000000u);
            chain_of[p] = ci;
        }
        a = srec[p];
        m = make_uint2(__ldg(&blen[idx]), __ldg(&matches[idx])); // gathered by input index (a separate sorted copy cost 16 B more per record)
    }
    // groups are contiguous: usually the whole warp shares one
    const u32 g0 = __shfl_sync(full, g, 0);
    if (__all_sync(full, g == g0)) {
        const u32 mn = __reduce_min_sync(full, idx);
        if (lane == 0 && g0 != NONE32) atomicMin(&grp_minidx[g0], mn);
    } else if (ok) {
        atomicMin(&grp_minidx[g], idx);
    }
    const u64 smv = m.y, sbk = m.x;
    const u32 peers = __match_any_sync(full, ci);
    const u32 leader = __ffs(peers) - 1;
    if (ok && __popc(peers) == 1) {
        atomicMin(&cd.qmin[ci], a.x); atomicMax(&cd.qmax[ci], a.y);
        atomicMin(&cd.tmin[ci], a.z); atomicMax(&cd.tmax[ci], a.w);
        atomicAdd((unsigned long long *)&cd.sum_matches[ci], (unsigned long long)smv);
        atomicAdd((unsigned long long *)&cd.sum_block[ci], (unsigned long long)sbk);
    }
    u32 todo = __ballot_sync(full, ok && __popc(peers) > 1 && lane == leader);
    while (todo) {
        const u32 Ld = __ffs(todo) - 1;
        todo &= todo - 1;
        const u32 pm = __shfl_sync(full, peers, Ld);
        const u32 cc = __shfl_sync(full, ci, Ld);
        const bool in = (pm >> lane) & 1;
        const u32 vqmin = __reduce_min_sync(full, in ? a.x : NONE32), vqmax = __reduce_max_sync(full, in ? a.y : 0u);
        const u32 vtmin = __reduce_min_sync(full, in ? a.z : NONE32), vtmax = __reduce_max_sync(full, in ? a.w : 0u);
        u64 vsm = in ? smv : 0, vsb = in ? sbk : 0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            vsm += __shfl_down_sync(full, vsm, o);
            vsb += __shfl_down_sync(full, vsb, o);
        }
        if (lane == 0) {
            atomicMin(&cd.qmin[cc], vqmin); atomicMax(&cd.qmax[cc], vqmax);
            atomicMin(&cd.tmin[cc], vtmin); atomicMax(&cd.tmax[cc], vtmax);
            atomicAdd((unsigned long long *)&cd.sum_matches[cc], (unsigned long long)vsm);
            atomicAdd((unsigned long long *)&cd.sum_block[cc], (unsigned long long)vsb);
        }
    }
}

// ---------------------------------------------------------------------------------------------
// chain table (dense, C rows)
// ---------------------------------------------------------------------------------------------
struct ChainTable {
    u32 *pos;              // sorted position of the head
    u32 *qid, *tid;
    u8 *fwd;
    u32 *qs, *qe, *ts, *te; // bounding box
    double *wid;           // weighted_identity
    u8 *pass;              // length/identity filter (paf_filter.rs:449-455)
    u32 *k;                // chain number (1-based) or 0
};

// ---------------------------------------------------------------------------------------------
// score_with_function, plane_sweep_exact.rs:29-86 (length = QUERY span on both axes)
// ---------------------------------------------------------------------------------------------
// `ln`: glibc_log (glibc_log.cuh: the host libm's bits) unless cuda_log is set (SWG_LOG_IMPL=cuda: CUDA's log(), a
// testing aid that stands in for "a host whose libm differs from the port").
__device__ __forceinline__ double ln_fn(double x, bool cuda_log) { return cuda_log ? log(x) : glibc_log(x); }
__device__ __forceinline__ double score_fn(int scoring, double identity, u32 qs, u32 qe, bool cuda_log = false) {
    double length = (double)(qe - qs);
    const double ninf = __longlong_as_double(0xFFF0000000000000LL);
    switch (scoring) {
    case 0: return identity <= 0.0 ? ninf : identity;
    case 1: return length <= 0.0 ? ninf : length;
    case 2:
    case 4: return (length <= 0.0 || identity <= 0.0) ? ninf : __dmul_rn(length, identity);
    default: return (length <= 0.0 || identity <= 0.0) ? ninf : __dmul_rn(identity, ln_fn(length, cuda_log));
    }
}
// weighted_identity of a chain, paf_filter.rs:896-913
__device__ __forceinline__ double chain_identity_fn(u64 total_length, u64 sum_block, u64 sum_matches, bool cuda_log, const double *host_lg = nullptr) {
    const u64 gap = total_length > sum_block ? total_length - sum_block : 0; // saturating_sub, :901
    double lg = 0.0;
    if (gap > 0) lg = host_lg ? *host_lg : fmax(ln_fn((double)gap, cuda_log), 0.0); // :902-906
    const double eff = __dadd_rn((double)sum_block, lg);
    return eff > 0.0 ? __ddiv_rn((double)sum_matches, eff) : 0.0;
}
// order-preserving map f64 -> u64, DESCENDING score = ascending key (MappingOrder::cmp, :183-194)
__device__ __forceinline__ u64 score_desc_key(double s) {
    u64 b = (u64)__double_as_longlong(s);
    if (b == 0x8000000000000000ULL) b = 0; // -0.0 == +0.0 under partial_cmp
    u64 asc = (b >> 63) ? ~b : (b | 0x8000000000000000ULL);
    return ~asc;
}
// query_overlap/target_overlap > thr, plane_sweep_exact.rs:113-144
__device__ __forceinline__ bool overlaps_more_than(u32 s1, u32 e1, u32 s2, u32 e2, double thr) {
    u32 os = max(s1, s2), oe = min(e1, e2);
    double ol = oe > os ? (double)(oe - os) : 0.0;
    double ml = fmin((double)(e1 - s1), (double)(e2 - s2));
    // The reference compares RN(ol / ml) with thr.  ol and ml are exact integers, so whenever ol is outside
    // thr * ml * (1 +- 2^-49) the rounded quotient is on the same side of thr as the exact one and the f64 division
    // (the most expensive instruction sequence of the sweep) is not needed; only the band in between divides.
    if (ml > 0.0 && thr >= 0.0 && thr < 1e300) {
        const double p = __dmul_rn(thr, ml);
        if (ol > __dmul_rn(p, 0x1.0000000000008p+0)) return true;
        if (ol < __dmul_rn(p, 0x1.ffffffffffff0p-1)) return false;
    }
    double ov = ml > 0.0 ? __ddiv_rn(ol, ml) : 0.0;
    return ov > thr;
}

// ---------------------------------------------------------------------------------------------
// General plane sweep (plane_sweep_exact.rs:197-433: event loop + mark_good) over groups whose items are sorted by
// (start, item).  Only the Begins are sorted: the End events come out of the active set itself — the next event
// position is min(next start, smallest end among the active items), which visits exactly the positions of the
// reference's (position, Begin-before-End) event list, in the same order, with half the sort volume.
// At a position: insert its Begins, remove every active item that ends there, then mark_good.
// good/flagged follow the closed form "kept <=> ever in the top-n at an evaluated position and never flagged
// overlapped".
// ---------------------------------------------------------------------------------------------
// Two scores this close can rank differently when the log comes from another libm (each side is within ~1 ulp of the
// other in the log, one more rounding in the product): the audit band of swg_stats.score_near_ties.
constexpr u64 NEAR_TIE_ULPS = 4;
// An exact tie counts too unless the two items also share the interval (duplicate records: same inputs, same score under
// any libm): equal device scores of DIFFERENT items may be unequal on the host.
__device__ __forceinline__ bool near_tie(u64 key_a, u32 start_a, u32 end_a, u64 key_b, u32 start_b, u32 end_b) {
    const u64 df = key_a > key_b ? key_a - key_b : key_b - key_a;
    return df <= NEAR_TIE_ULPS && !(df == 0 && start_a == start_b && end_a == end_b);
}
struct SweepItem { // per item, in (group, start, item) order, so that a group is one contiguous stream
    u64 skey;  // score_desc_key of the item
    u32 start; // axis interval of the item
    u32 end;
};
struct ActEntry {
    u64 skey; // score_desc_key
    u32 start, end;
    u32 item, pad;
};
__device__ __forceinline__ bool act_less(const ActEntry &a, const ActEntry &b) {
    if (a.skey != b.skey) return a.skey < b.skey;
    if (a.start != b.start) return a.start < b.start;
    return a.item < b.item;
}

// n_keep == 1 (the 1:1 modes): the same result without walking a group sequentially — ONE THREAD PER ITEM.
// After the events of a position p the active set is S(p) = { k : start_k <= p < end_k }.  Item m is marked good iff it
// is the best of S(p) at some event position p in [start_m, end_m), and flagged iff at some such p it is not the best
// and overlaps the best by more than thr.  Every member of S(p) for such p intersects m's span, so the thread only
// looks at its neighbours in start order: to the right while start_k < end_m, to the left while some item at or left of k
// still reaches start_m — one load of the group's running maximum of the interval ends (pmax[k] = max end over the group's
// items up to k, scan_segmax): on collinear data the scan stops after a step or two however long the longest item of the group
// is.  S(p) changes only at the starts and ends of those neighbours.  Groups where a scan gets long (deep piles, one very long item)
// are listed and go through the position-parallel tree sweep (sweep_tree.cuh), which decides the keep bytes of their items.
constexpr u32 SWF_LEFT = 48, SWF_RIGHT = 48;
// the verdict of one item (sorted position u): everything k_sweep_flat1's header describes
__device__ __forceinline__ void sweep_flat1_item(u32 u, const u32 *__restrict__ sitem, const SweepItem *__restrict__ sdata, const u32 *__restrict__ gid,
                                                 const u32 *__restrict__ gstart, const u32 *__restrict__ pmax, u32 n_groups, u32 n_sorted, double thr,
                                                 u8 *__restrict__ keep, u32 *gflag, u32 *big_list, u32 *big_count, u64 *ctr, u32 scan_limit) {
    const u32 g = gid[u];
    const u32 gs = gstart[g], ge = (g + 1 < n_groups) ? gstart[g + 1] : n_sorted;
    const u32 item = sitem[u];
    const SweepItem me = sdata[u];
    bool big = scan_limit == 0;
    u32 lo = u, hi = u;
    for (u32 k = u, steps = 0; k > gs && !big;) {
        k--;
        if (pmax[k] <= me.start) break; // nothing at or left of k reaches start_m
        const SweepItem a = sdata[k];
        if (a.end > me.start) lo = k;
        if (++steps > scan_limit) { big = true; break; }
    }
    u32 near = 0;
    for (u32 k = u + 1; k < ge && !big; k++) {
        const SweepItem a = sdata[k];
        if (a.start >= me.end) break;
        hi = k;
        near += near_tie(a.skey, a.start, a.end, me.skey, me.start, me.end); // near-tie audit, each co-active pair once
        if (k - u > scan_limit) big = true;
    }
    if (big) {
        if (atomicExch(&gflag[g], 1u) == 0) big_list[atomicAdd(big_count, 1u)] = g;
        return;
    }
    if (near) atomicAdd((unsigned long long *)&ctr[C_NEAR_TIES], (unsigned long long)near);
    bool is_good = false, is_flag = false;
    const bool want_flag = thr < 1.0;
    auto eval = [&](u32 p) {
        u64 bkey = me.skey;
        u32 bstart = me.start, bend = me.end, bpos = u;
        for (u32 k = lo; k <= hi; k++) {
            if (k == u) continue;
            const SweepItem a = sdata[k];
            if (a.start <= p && p < a.end) {
                bool less = a.skey < bkey || (a.skey == bkey && a.start < bstart);
                if (!less && a.skey == bkey && a.start == bstart) less = sitem[k] < sitem[bpos];
                if (less) { bkey = a.skey; bstart = a.start; bend = a.end; bpos = k; }
            }
        }
        if (bpos == u) is_good = true;
        else if (want_flag && !is_flag) is_flag = overlaps_more_than(me.start, me.end, bstart, bend, thr);
    };
    eval(me.start);
    for (u32 k = lo; k <= hi && !is_flag; k++) {
        if (is_good && !want_flag) break;
        if (k == u) continue;
        const SweepItem a = sdata[k];
        if (k > u && a.start > me.start) eval(a.start);
        if (a.end > me.start && a.end < me.end) eval(a.end);
    }
    if (is_good && !is_flag) keep[item] = 1;
}
// First pass, 1024 items per CTA: an item alone in its span — nothing to its left reaches its start, its right neighbour starts at
// or after its end: nine in ten on collinear data — is the best of every active set it is in: kept, no neighbour scan.  The others
// are LISTED (one counter atomic per CTA) and judged by k_sweep_flat1_rest with all lanes busy (judging them in place ran at 12 of
// 32 threads per instruction).
__global__ void __launch_bounds__(256)
k_sweep_flat1(const u32 *__restrict__ sitem, const SweepItem *__restrict__ sdata, const u32 *__restrict__ gid, const u32 *__restrict__ gstart,
              const u32 *__restrict__ pmax, u32 n_groups, u32 n_sorted, u8 *__restrict__ keep, u32 *__restrict__ rest, u32 *rest_count, u32 scan_limit) {
    __shared__ u32 s_w[8][4];
    __shared__ u32 s_base;
    const u32 lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const u32 base = blockIdx.x * 1024;
    bool f[4];
    u32 m[4];
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const u32 u = base + k * 256 + threadIdx.x;
        f[k] = false;
        if (u < n_sorted) {
            const u32 g = gid[u];
            const u32 gs = gstart[g], ge = (g + 1 < n_groups) ? gstart[g + 1] : n_sorted;
            if (ge - gs <= 1) keep[sitem[u]] = 1; // a single interval: kept (plane_sweep_exact.rs:274-276)
            else {
                const SweepItem me = sdata[u];
                if (me.end > me.start) { // (zero length: its End follows its Begin at the same position, never evaluated: keep stays 0)
                    const bool alone = scan_limit != 0 && (u == gs || pmax[u - 1] <= me.start) && (u + 1 == ge || sdata[u + 1].start >= me.end);
                    if (alone) keep[sitem[u]] = 1;
                    else f[k] = true;
                }
            }
        }
        m[k] = __ballot_sync(0xFFFFFFFFu, f[k]);
        if (lane == 0) s_w[warp][k] = __popc(m[k]);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        u32 tot = 0;
        for (int k = 0; k < 4; k++)
            for (int w = 0; w < 8; w++) { const u32 t = s_w[w][k]; s_w[w][k] = tot; tot += t; }
        s_base = tot ? atomicAdd(rest_count, tot) : 0;
    }
    __syncthreads();
    const u32 lt = (1u << lane) - 1;
#pragma unroll
    for (int k = 0; k < 4; k++)
        if (f[k]) rest[s_base + s_w[warp][k] + __popc(m[k] & lt)] = base + k * 256 + threadIdx.x;
}
__global__ void __launch_bounds__(256)
k_sweep_flat1_rest(const u32 *__restrict__ rest, const u32 *__restrict__ rest_count, const u32 *__restrict__ sitem, const SweepItem *__restrict__ sdata,
                   const u32 *__restrict__ gid, const u32 *__restrict__ gstart, const u32 *__restrict__ pmax, u32 n_groups, u32 n_sorted, double thr,
                   u8 *__restrict__ keep, u32 *gflag, u32 *big_list, u32 *big_count, u64 *ctr, u32 scan_limit) {
    const u32 n = *rest_count;
    for (u32 x = blockIdx.x * blockDim.x + threadIdx.x; x < n; x += gridDim.x * blockDim.x)
        sweep_flat1_item(rest[x], sitem, sdata, gid, gstart, pmax, n_groups, n_sorted, thr, keep, gflag, big_list, big_count, ctr, scan_limit);
}

// sort keys of the included items: (group << pbits) | start, payload = item (pbits == 64: the start alone, the group id
// is applied by a second stable sort); one counter atomic per CTA
__global__ void __launch_bounds__(256) k_sweep_keys(u32 n_items, const u8 *__restrict__ include, u8 include_mask, const u64 *__restrict__ gkey,
                                                    int pbits, const u32 *__restrict__ it_start, u64 *__restrict__ ek, u32 *__restrict__ ev,
                                                    u64 *__restrict__ n_included) {
    u32 mine = 0; // grid-stride: one counter atomic per CTA of a grid of a few thousand (78 k same-address atomics cost ~80 us)
    for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < n_items; i += gridDim.x * blockDim.x) {
        const bool inc = include ? (include[i] & include_mask) != 0 : true;
        ek[i] = inc ? ((pbits >= 64 ? 0 : (gkey[i] << pbits)) | (u64)it_start[i]) : NONE64;
        ev[i] = i;
        mine += inc ? 1u : 0u;
    }
    const int slots[1] = {0};
    const u32 vals[1] = {mine};
    block_count_add<1>(n_included, slots, vals);
}

// One warp per group, for the groups whose pile is deeper than the per-thread array of k_sweep_small.  The active set
// is a rank-ordered array (score desc, start asc, item asc) in a per-group slice of global scratch.
__global__ void __launch_bounds__(128)
k_sweep_groups(const u32 *__restrict__ sitem, const SweepItem *__restrict__ sdata, const u32 *__restrict__ gstart, u32 n_groups, u32 n_sorted,
               u64 n_keep, double thr, ActEntry *act, u8 *good, u8 *flagged, const u32 *__restrict__ work,
               const u32 *__restrict__ n_work_ptr, u32 *group_counter, u64 *ctr) {
    const u32 full = 0xFFFFFFFFu;
    const u32 lane = lane_id();
    const u32 n_work = *n_work_ptr;
    while (true) {
        u32 w = 0;
        if (lane == 0) w = atomicAdd(group_counter, 1u);
        w = __shfl_sync(full, w, 0);
        if (w >= n_work) break;
        const u32 g = work[w];
        const u32 es = gstart[g], ee = (g + 1 < n_groups) ? gstart[g + 1] : n_sorted;
        if (ee - es <= 1) { // plane_sweep_exact.rs:274-276
            if (lane == 0) good[sitem[es]] = 1;
            continue;
        }
        ActEntry *A = act + es;
        u32 size = 0;
        u32 e = es;
        while (e < ee || size > 0) {
            // the position of the next event
            u32 mn = NONE32;
            for (u32 b = lane; b < size; b += 32) mn = min(mn, A[b].end);
            mn = __reduce_min_sync(full, mn);
            u32 cur = mn;
            if (e < ee) cur = min(cur, sdata[e].start);
            bool ends_here = size > 0 && mn == cur;
            // Begins at cur
            while (e < ee) {
                const SweepItem d = sdata[e];
                if (d.start != cur) break;
                ActEntry x;
                x.skey = d.skey; x.start = d.start; x.end = d.end; x.item = sitem[e]; x.pad = 0;
                ends_here |= d.end == cur;
                // position of x in A: number of entries ordered before it
                u32 cnt = 0;
                for (u32 b = lane; b < size; b += 32) cnt += act_less(A[b], x) ? 1 : 0;
                cnt = __reduce_add_sync(full, cnt);
                // near-tie audit: neighbours whose score key differs by <= 2 ulp but is not equal
                if (lane == 0) {
                    u32 near = 0;
                    if (cnt > 0) near += near_tie(x.skey, x.start, x.end, A[cnt - 1].skey, A[cnt - 1].start, A[cnt - 1].end);
                    if (cnt < size) near += near_tie(x.skey, x.start, x.end, A[cnt].skey, A[cnt].start, A[cnt].end);
                    if (near) atomicAdd((unsigned long long *)&ctr[C_NEAR_TIES], (unsigned long long)near);
                }
                // shift [cnt, size) up by one, from the top, 32 at a time
                for (u32 hi = size; hi > cnt;) {
                    u32 lo = hi > cnt + 32 ? hi - 32 : cnt;
                    u32 b = lo + lane;
                    ActEntry t;
                    bool mv = b < hi;
                    if (mv) t = A[b];
                    __syncwarp();
                    if (mv) A[b + 1] = t;
                    __syncwarp();
                    hi = lo;
                }
                if (lane == 0) A[cnt] = x;
                size++;
                __syncwarp();
                e++;
            }
            // Ends at cur: stable compaction of the entries that stay
            if (ends_here) {
                u32 out = 0;
                for (u32 lo = 0; lo < size; lo += 32) {
                    const u32 b = lo + lane;
                    ActEntry t;
                    const bool in = b < size;
                    if (in) t = A[b];
                    const bool kp = in && t.end != cur;
                    const u32 m = __ballot_sync(full, kp);
                    if (kp) A[out + __popc(m & lanemask_lt())] = t; // destination <= source, earlier chunks are consumed
                    out += __popc(m);
                    __syncwarp();
                }
                size = out;
            }
            if (size == 0) continue;
            // mark_good (plane_sweep_exact.rs:197-259)
            const u32 top = (u64)size <= n_keep ? size : (u32)n_keep;
            for (u32 b = lane; b < top; b += 32) good[A[b].item] = 1;
            if (thr < 1.0 && top < size) {
                for (u32 b = top + lane; b < size; b += 32) {
                    const ActEntry me = A[b];
                    if (flagged[me.item]) continue;
                    for (u32 t = 0; t < top; t++) {
                        if (overlaps_more_than(me.start, me.end, A[t].start, A[t].end, thr)) { flagged[me.item] = 1; break; }
                    }
                }
            }
            __syncwarp();
        }
        __syncwarp();
    }
}

// The same sweep, ONE THREAD PER GROUP, for the ordinary case (a (sequence, partner-genome) group of ~10^2 intervals
// with a pile depth of a few): the active set lives in a small per-thread array; a group whose depth exceeds
// SW_DEPTH is handed to the warp kernel above (good/flagged are monotone, so the redo is idempotent).
#ifndef SWG_SW_DEPTH
#define SWG_SW_DEPTH 12
#endif
constexpr int SW_DEPTH = SWG_SW_DEPTH;
__global__ void __launch_bounds__(128)
k_sweep_small(const u32 *__restrict__ sitem, const SweepItem *__restrict__ sdata, const u32 *__restrict__ gstart, u32 n_groups, u32 n_sorted,
              u64 n_keep, double thr, u8 *good, u8 *flagged, u32 *big_list, u32 *big_count, u32 *group_counter, u64 *ctr) {
    const u32 full = 0xFFFFFFFFu;
    bool active = false, exhausted = false;
    u32 g = 0, e = 0, ee = 0, size = 0;
    u32 mn = NONE32; // smallest end among the active entries
    u32 chk = 0;     // n_keep == 1: bit b = entry b has been compared with the current best entry (an overlap never changes)
    u64 a_key[SW_DEPTH];
    u32 a_start[SW_DEPTH], a_end[SW_DEPTH], a_item[SW_DEPTH]; // a_item: item * 4 | (flagged << 1) | good-written
    while (true) {
        const u32 need = __ballot_sync(full, !active && !exhausted);
        if (need) {
            const u32 leader = __ffs(need) - 1;
            u32 base = 0;
            if (lane_id() == leader) base = atomicAdd(group_counter, (u32)__popc(need));
            base = __shfl_sync(full, base, leader);
            if (!active && !exhausted) {
                g = base + __popc(need & lanemask_lt());
                if (g >= n_groups) exhausted = true;
                else {
                    e = gstart[g];
                    ee = (g + 1 < n_groups) ? gstart[g + 1] : n_sorted;
                    if (ee - e <= 1) good[sitem[e]] = 1; // a single interval: kept (plane_sweep_exact.rs:274-276)
                    else { active = true; size = 0; mn = NONE32; chk = 0; }
                }
            }
        }
        if (__all_sync(full, exhausted && !active)) break;
        if (active) {
            // one event position per iteration: min(next start, smallest active end); its Begins, its Ends, then mark_good
            u32 cur = mn;
            bool have = e < ee;
            SweepItem d;
            if (have) { d = sdata[e]; cur = min(cur, d.start); }
            bool ends_here = size > 0 && mn == cur;
            bool overflow = false;
            while (have && d.start == cur) { // Begin: insert in (score desc, start asc, item asc) order
                if (size == SW_DEPTH) { overflow = true; break; }
                const u32 item = sitem[e];
                u32 pos = size;
                while (pos > 0) {
                    const u32 q = pos - 1;
                    const bool less = a_key[q] < d.skey || (a_key[q] == d.skey && (a_start[q] < d.start || (a_start[q] == d.start && (a_item[q] >> 2) < item)));
                    if (less) break;
                    a_key[pos] = a_key[q]; a_start[pos] = a_start[q]; a_end[pos] = a_end[q]; a_item[pos] = a_item[q];
                    pos--;
                }
                a_key[pos] = d.skey; a_start[pos] = d.start; a_end[pos] = d.end; a_item[pos] = item << 2;
                u32 near = 0; // near-tie audit: neighbours whose score key differs by <= 2 ulp but is not equal
                if (pos > 0) near += near_tie(d.skey, d.start, d.end, a_key[pos - 1], a_start[pos - 1], a_end[pos - 1]);
                if (pos < size) near += near_tie(d.skey, d.start, d.end, a_key[pos + 1], a_start[pos + 1], a_end[pos + 1]);
                if (near) atomicAdd((unsigned long long *)&ctr[C_NEAR_TIES], (unsigned long long)near);
                size++;
                chk = pos == 0 ? 0u : ((chk & ((1u << pos) - 1)) | ((chk >> pos) << (pos + 1)));
                mn = min(mn, d.end);
                ends_here |= d.end == cur;
                e++;
                have = e < ee;
                if (have) d = sdata[e];
            }
            if (overflow) {
                big_list[atomicAdd(big_count, 1u)] = g; // pile deeper than SW_DEPTH: the warp kernel redoes this group
                active = false;
            } else {
                if (ends_here) { // End: remove every entry that ends here, keeping the order of the others
                    u32 o = 0, nchk = 0;
                    mn = NONE32;
                    const bool best_leaves = a_end[0] == cur;
                    for (u32 b = 0; b < size; b++) {
                        const u32 en = a_end[b];
                        if (en != cur) {
                            if (o != b) { a_key[o] = a_key[b]; a_start[o] = a_start[b]; a_end[o] = en; a_item[o] = a_item[b]; }
                            nchk |= ((chk >> b) & 1u) << o;
                            mn = min(mn, en);
                            o++;
                        }
                    }
                    chk = best_leaves ? 0u : nchk;
                    size = o;
                }
                if (size > 0) { // mark_good, plane_sweep_exact.rs:197-259
                    const u32 top = (u64)size <= n_keep ? size : (u32)n_keep;
                    for (u32 b = 0; b < top; b++)
                        if (!(a_item[b] & 1)) { good[a_item[b] >> 2] = 1; a_item[b] |= 1; }
                    if (thr < 1.0) {
                        if (top == 1) { // every entry meets a given best entry once
                            const u32 s0 = a_start[0], e0 = a_end[0];
                            for (u32 b = 1; b < size; b++) {
                                if ((a_item[b] & 2) || ((chk >> b) & 1u)) continue;
                                chk |= 1u << b;
                                if (overlaps_more_than(a_start[b], a_end[b], s0, e0, thr)) {
                                    flagged[a_item[b] >> 2] = 1;
                                    a_item[b] |= 2;
                                }
                            }
                        } else {
                            for (u32 b = top; b < size; b++) {
                                if (a_item[b] & 2) continue;
                                for (u32 t = 0; t < top; t++) {
                                    if (overlaps_more_than(a_start[b], a_end[b], a_start[t], a_end[t], thr)) {
                                        flagged[a_item[b] >> 2] = 1;
                                        a_item[b] |= 2;
                                        break;
                                    }
                                }
                            }
                        }
                    }
                }
                if (e >= ee && size == 0) active = false;
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// plane_sweep_core::plane_sweep (src/plane_sweep_core.rs:80-201) — the secondary Interval API.  Different
// semantics from plane_sweep_exact on purpose: the n best active intervals are marked after EVERY Begin event,
// Ends only remove, and the overlap rule is a greedy pass over the marked set in score order.  One warp
// (library / test API, not on the filter pipeline).
// ---------------------------------------------------------------------------------------------
struct CoreEntry { u64 key; u32 idx; u32 pad; }; // key = order-preserving image of -(score bits as i64)
__device__ __forceinline__ u64 core_key(double score) {
    const i64 k = (i64)(0ull - (u64)__double_as_longlong(score)); // wrapping negation like release Rust
    return (u64)k ^ 0x8000000000000000ULL;
}
__global__ void __launch_bounds__(32)
k_sweep_core_mark(const u32 *__restrict__ ev /* idx*2+type in (pos,type,idx) order */, u32 n_ev, const double *__restrict__ score,
                  u64 max_keep, CoreEntry *A, u8 *marked) {
    const u32 full = 0xFFFFFFFFu;
    const u32 lane = lane_id();
    u32 size = 0;
    for (u32 e = 0; e < n_ev; e++) {
        const u32 idx = ev[e] >> 1;
        const bool is_end = ev[e] & 1;
        CoreEntry x;
        x.key = core_key(score[idx]); x.idx = idx; x.pad = 0;
        u32 cnt = 0;
        for (u32 b = lane; b < size; b += 32) cnt += (A[b].key < x.key || (A[b].key == x.key && A[b].idx < x.idx)) ? 1 : 0;
        cnt = __reduce_add_sync(full, cnt);
        if (!is_end) {
            for (u32 hi = size; hi > cnt;) {
                u32 lo = hi > cnt + 32 ? hi - 32 : cnt;
                u32 b = lo + lane;
                CoreEntry t;
                bool mv = b < hi;
                if (mv) t = A[b];
                __syncwarp();
                if (mv) A[b + 1] = t;
                __syncwarp();
                hi = lo;
            }
            if (lane == 0) A[cnt] = x;
            size++;
            __syncwarp();
            const u32 top = (u64)size <= max_keep ? size : (u32)max_keep; // mark_best, :152-164
            for (u32 b = lane; b < top; b += 32) marked[A[b].idx] = 1;
        } else {
            for (u32 lo = cnt + 1; lo < size; lo += 32) {
                u32 b = lo + lane;
                CoreEntry t;
                bool mv = b < size;
                if (mv) t = A[b];
                __syncwarp();
                if (mv) A[b - 1] = t;
                __syncwarp();
            }
            size--;
        }
        __syncwarp();
    }
}
// filter_by_overlap (:167-201): candidates in score-descending order, keep those that do not overlap a kept one
__global__ void __launch_bounds__(32)
k_sweep_core_greedy(const u32 *__restrict__ order, u32 n_c, const u32 *__restrict__ begin, const u32 *__restrict__ end, double thr,
                    u32 *accepted, u32 *n_accepted) {
    const u32 full = 0xFFFFFFFFu;
    const u32 lane = lane_id();
    u32 na = 0;
    for (u32 t = 0; t < n_c; t++) {
        const u32 i = order[t];
        const u32 bi = begin[i], ei = end[i];
        bool hit = false;
        for (u32 a = lane; a < na && !hit; a += 32) {
            const u32 k = accepted[a];
            const u32 os = max(bi, begin[k]), oe = min(ei, end[k]);
            if (os < oe) {
                const u32 ml = min(ei - bi, end[k] - begin[k]);
                hit = __ddiv_rn((double)(oe - os), (double)ml) > thr;
            }
        }
        if (!__any_sync(full, hit)) {
            if (lane == 0) accepted[na] = i;
            na++;
        }
        __syncwarp();
    }
    if (lane == 0) *n_accepted = na;
}

} // namespace swg

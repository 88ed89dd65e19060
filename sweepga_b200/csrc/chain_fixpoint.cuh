// chain_fixpoint.cuh — best-buddy chaining of HUGE (query,target,strand) groups as a parallel fixed-point iteration.
//
// The reference (src/paf_filter.rs:784-851) walks the positions i of a group in order; position i picks the successor j
// that minimises d(i,j) among the candidates with d(i,j) < best_pred_score[j], and best_pred_score[j] is the d of the LAST
// position before i that picked j (every successful pick lowers it).  So
//
//     pick(i) = first arg-min_j { d(i,j) : d(i,j) < B(i,j) },   B(i,j) = min { d(i',j) : i' < i, pick(i') = j }      (*)
//
// and pick(i) depends only on the picks of smaller positions: (*) has exactly one solution, the reference's.  One thread
// or warp walking a 25 M-mapping centromeric pile pays a memory round trip per step (k_chain_resolve_warp: ~1.3 us per
// mapping); here ALL positions are evaluated against a snapshot of the picks and the evaluation is repeated until nothing
// changes.  By induction on i the positions below the first wrong one stay correct and that one becomes correct in the
// next round, so the iteration ends in the reference's picks; measured on the configs[4] piles it needs 6 rounds for a
// 100 k group, 14 for a 500 k group and 56 for the two 25 M groups of the full configuration (1.45 s for the whole filter
// call), and the number of positions that have to be re-evaluated shrinks geometrically.
//
// A round:
//   1. snapshot: picker lists per successor j (CSR) in position order — the positions sorted by their pick, stable — with the
//      picker d stored as prefix minima; per successor one 32 B word: the smallest d over all pickers of j, minpi[j] = the
//      first picker holding it, firstp[j] = the first picker at all and its d, the list range.  "d < B(i,j)?" is answered from
//      that word in all but a few cases (fx_eligible_packed), else by one binary search over the list.
//   2. k_fx_check_warp (lane per position, X(i) lists read by whole warps; a position is skipped outright when no picker list
//      among the successors it can depend on — up to xhi[i] = max(pick(i), X(i)) — changed in the last round: dirty blocks of
//      512 successors and their prefix counts; an entry whose successor's own list did not change — one bit per successor —
//      keeps its verdict): position i must be re-evaluated iff its pick is now blocked (an earlier picker
//      of the same j with d' <= d) or one of the candidates that rank BEFORE its pick — X(i), all of them ineligible when
//      the pick was made, remembered explicitly with their d — has become eligible.  This test is exact: a position whose pick
//      stands and whose X(i) is still blocked would pick the same j again.
//   3. k_fx_recompute (warp per listed position): the search in target-bucket order (fx_bucket_pass: the group's positions
//      once more by (bucket of the target coordinate the gap rule tests, position); buckets visited outwards from the position's
//      own, pruned outward scans inside a bucket) with eligibility against the snapshot.  The blocked candidates the search meets
//      while they still beat the lane's best are recorded in shared memory — a superset of X(i), filtered against the final pick
//      (fx_filter_seen); only if that record overflows, a second pruned pass collects X(i).
// A huge group whose picks have not settled after SWG_FIXPOINT_MAX_ROUNDS rounds goes to the sequential walk after all;
// SWG_FIXPOINT_VERIFY=1 re-evaluates every position from scratch against the final picks (0 of 50 M change on configs[4]).
// Round 0 evaluates every position against the empty snapshot: the unconstrained arg-min (X(i) is empty there by definition).
// After the last round pred[j] = the last picker of j, roots by pointer jumping (union_find.rs:25-41: the root of a set is
// its head), results scattered back to the sorted positions.  Everything runs in the compact index space k of the positions
// that belong to huge groups (groups stay contiguous there, so successor offsets carry over).
#pragma once

namespace swg {

struct t_fx_init; struct t_fx_skey; struct t_fx_pm; struct t_fx_bkey; struct t_fx_brec; struct t_fx_count; struct t_fx_all; struct t_fx_pred; struct t_fx_jump; struct t_fx_scatter;

constexpr u32 FX_XCAP = 1024;     // blocked candidates remembered per position; a position with more is re-evaluated every round
constexpr u16 FX_XOVER = 0xFFFF; // xcnt value of such a position
constexpr u32 FX_REV = 0x80000000u; // gend bit: the group is a '-' strand group
constexpr int FX_DB = 9;            // dirty blocks of 512 successors

struct FxArrays {
    u32 n;             // positions in huge groups
    uint4 *rec;        // (qs, qe, ts, te)
    u32 *gend;         // end of the position's group (k-space) | FX_REV
    u32 *pick;         // current pick (k-space), NONE32 = none
    u64 *pd;           // d of the current pick
    u32 *cnt, *off;    // picker lists: off[j] .. off[j+1], in position order
    u32 *minpi;        // the first picker of j that has the smallest d over all pickers of j
    u32 *firstp;       // the first picker of j at all (NONE32: nobody)
    u32 *li;           // picker position
    u64 *ld;           // the smallest picker d of the list up to and including this entry
    u32 force_collect; // testing aid (SWG_FX_FORCE_COLLECT=1): X(i) always from the separate collecting pass
    u32 *xoff;         // X(i) lives at pool[xoff .. xoff + xcnt)
    u16 *xcnt, *xcap;
    u32 *pool;
    u64 *pool_d;       // d(i, x) of every pool entry (k_fx_check_warp then needs no record gather)
    unsigned long long *pool_top; // 64-bit: refused requests keep counting and must never wrap into live slots
    u32 pool_cap;
    u32 *list;         // positions to re-evaluate this round
    u32 *xhi;          // largest position in {pick(i)} U X(i) (i itself if there is none): how far i's verdict can depend
    u32 *dirty, *dps;  // per block of successors: some picker list in it changed in the last round; prefix counts of that
    u32 use_dirty;     // 0: check every position (first round)
    u32 *dbits, *dbits_w; // one bit per successor: its picker list changed in the last round (read by k_fx_check_warp) / in this one
    u32 *ctrs;         // [0] list length, [1] picks changed this round, [2] recompute work counter, [3] slots refused (pool full)
    // target-bucket order (fx_bucket_pass): the positions of every huge group once more, ordered by (group, target bucket, k)
    u32 *hg;           // dense number of the position's huge group
    uint4 *snap;       // 32 B (one sector) per successor: [2j] = (smallest picker d lo, hi, minpi, firstp), [2j+1] = (d of the first picker lo, hi, off[j], list length)
    uint2 *bq;         // (query_start, t') of the entries in bucket order: all the gap rule reads of a candidate
    u32 *bk;           // their positions k
    u32 *dir;          // dir[hg * dirD + b] .. dir[hg * dirD + b + 1]: the entries of bucket b of the group
    u32 dirD;          // directory entries per group (buckets + 1)
    int bshift;        // bucket of a target coordinate x: x >> bshift
};

// is some picker of j before position i with d' <= d?  (the caller knows that the list is not empty)
// Position order + prefix minima: the last picker before i answers for all of them.
__device__ __forceinline__ bool fx_list_blocks(const FxArrays &f, u32 i, u32 j, u64 d, u32 a = NONE32, u32 b = NONE32) {
    if (a == NONE32) { a = f.off[j]; b = f.off[j + 1]; }
    u32 lo = a, hi = b;
    while (hi - lo > 4) {
        const u32 mid = (lo + hi) >> 1;
        if (f.li[mid] < i) lo = mid + 1; else hi = mid;
    }
    while (lo < hi && f.li[lo] < i) lo++;
    return lo > a && f.ld[lo - 1] <= d;
}
// smallest d over the pickers of j that precede position i, compared with d: true iff d < B(i,j)
// (callers have established that d is not below the smallest d over all pickers of j: if the picker that holds that minimum
// precedes i, that settles it)
__device__ __forceinline__ bool fx_eligible(const FxArrays &f, u32 i, u32 j, u64 d, u32 mi /* = minpi[j] */) {
    if (mi < i) return false;
    if (mi == i) return true; // i itself holds the minimum and is the first to: every earlier picker has a larger d
    if (f.firstp[j] >= i) return true; // nobody picks j before i (ncu: the list walk below was 30 % of the stall samples of round 1)
    return !fx_list_blocks(f, i, j, d);
}
// The verdict from the packed snapshot of j.  The holder of the smallest d and the first picker settle most cases; between them
// (first picker < i < holder of the minimum) the first picker's own d settles a list of two, and only longer lists are searched
// — the second word of the snapshot lies in the sector the first came from.
__device__ __forceinline__ bool fx_eligible_packed(const FxArrays &f, u32 i, u32 j, u64 d, u32 mi, u32 fp) {
    if (mi < i) return false;
    if (mi == i || fp >= i) return true;
    const uint4 s2 = f.snap[2 * (size_t)j + 1];
    const u64 fd = ((u64)s2.y << 32) | s2.x;
    if (fd <= d) return false;
    if (s2.w <= 2) return true;
    return !fx_list_blocks(f, i, j, d, s2.z, s2.z + s2.w);
}
struct FxExtra {
    FxArrays f;
    u32 i;
    u32 *seen, *n_seen; // shared memory of the warp: the blocked candidates met by the search (a superset of X(i))
    // the verdict from the packed snapshot word of j (mi = minpi[j], fp = firstp[j]); callers have established that d is not
    // below the smallest d over all pickers of j
    __device__ __forceinline__ bool packed(u32 j, u64 d, u32 mi, u32 fp) const {
        const bool el = fx_eligible_packed(f, i, j, d, mi, fp);
        if (!el) { // it beat the lane's best so far and is blocked: the only kind of candidate that can belong to X(i)
            const u32 o = atomicAdd(n_seen, 1u);
            if (o < FX_XCAP) seen[o] = j;
        }
        return el;
    }
};

// Round 0 for the positions whose window ends within the next BB_LINEAR successors — every position of a chromosome-scale group of
// collinear mappings, which is huge and sparse: one thread scans them in order (the unconstrained arg-min, first minimal j), no warp
// search.  A position whose window goes on (a pile) is listed for k_fx_recompute.
__global__ void __launch_bounds__(256) k_fx_round0_linear(FxArrays f, u64 G) {
    const u32 k = blockIdx.x * blockDim.x + threadIdx.x;
    bool more = false;
    if (k < f.n) {
        const uint4 a = f.rec[k];
        const u32 ge = f.gend[k];
        u64 bd;
        u32 bj;
        bb_best_successor<false>(f.rec, nullptr, k, ge & ~FX_REV, a, !(ge & FX_REV), G, G / 5, bd, bj, nullptr, &more);
        if (!more) {
            f.pick[k] = bj;
            f.pd[k] = bd;
            f.xhi[k] = bj != NONE32 ? bj : k;
        }
    }
    const u32 m = __ballot_sync(0xFFFFFFFFu, more);
    if (m) {
        u32 base = 0;
        const u32 leader = __ffs(m) - 1;
        if (lane_id() == leader) base = atomicAdd(&f.ctrs[0], (u32)__popc(m));
        base = __shfl_sync(0xFFFFFFFFu, base, leader);
        if (more) f.list[base + __popc(m & lanemask_lt())] = k;
    }
}

// step 2: does position k have to be re-evaluated against the new snapshot?  A lane first judges its own position (skip tests, its
// pick); the X(i) lists that still have to be looked at are then taken one at a time by all 32 lanes — coalesced reads of the pool
// instead of 32 private strided walks (at 50 M the pool holds 2.7 * 10^9 entries and a thread-per-position loop moved them at a tenth
// of the HBM rate) — and an entry whose successor's picker list did not change keeps last round's verdict without a further load.
__global__ void __launch_bounds__(256) k_fx_check_warp(FxArrays f, u64 G) {
    const u32 full = 0xFFFFFFFFu;
    const u32 lane = lane_id();
    const u32 k = blockIdx.x * blockDim.x + threadIdx.x;
    const bool bits = f.use_dirty != 0;
    bool need = false, scan_x = false;
    u32 xc = 0, xo = 0;
    if (k < f.n) {
        const u16 c = f.xcnt[k];
        const u32 j = f.pick[k];
        bool untouched = false;
        if (c != FX_XOVER && f.use_dirty) {
            const u32 hi = f.xhi[k];
            untouched = hi <= k || f.dps[(hi >> FX_DB) + 1] == f.dps[(k + 1) >> FX_DB];
        }
        if (c == FX_XOVER) need = true;
        else if (!untouched) {
            if (j != NONE32 && f.off[j + 1] - f.off[j] > 1 && (!bits || (f.dbits[j >> 5] >> (j & 31) & 1))) need = !fx_eligible(f, k, j, f.pd[k], f.minpi[j]);
            if (!need && c) { scan_x = true; xc = c; xo = f.xoff[k]; }
        }
    }
    u32 todo = __ballot_sync(full, scan_x);
    while (todo) {
        const u32 t = __ffs(todo) - 1;
        todo &= todo - 1;
        const u32 cnt = __shfl_sync(full, xc, t), base = __shfl_sync(full, xo, t), kt = k - lane + t;
        bool hit = false;
        for (u32 q0 = 0; q0 < cnt && !hit; q0 += 32) {
            const u32 q = q0 + lane;
            bool e = false;
            if (q < cnt) {
                const u32 jx = f.pool[base + q];
                if (!bits || (f.dbits[jx >> 5] >> (jx & 31) & 1)) {
                    const u64 d = f.pool_d[base + q];
                    const uint4 sn = f.snap[2 * (size_t)jx];
                    const u64 mp = ((u64)sn.y << 32) | sn.x;
                    e = d < mp || fx_eligible_packed(f, kt, jx, d, sn.z, sn.w);
                }
            }
            hit = __any_sync(full, e);
        }
        if (hit && lane == t) need = true;
    }
    const u32 m = __ballot_sync(full, need);
    if (m) {
        u32 base = 0;
        const u32 leader = __ffs(m) - 1;
        if (lane == leader) base = atomicAdd(&f.ctrs[0], (u32)__popc(m));
        base = __shfl_sync(full, base, leader);
        if (need) f.list[base + __popc(m & lanemask_lt())] = k;
    }
}

// X(i) = the valid candidates that rank before (bd, bj): appended to xs[0 .. FX_XCAP), returns how many there are
__device__ __forceinline__ u32 fx_collect_chunk(const uint4 &a, bool fwd, u64 G, u64 G5, u64 bd, u32 bj, u32 j, bool inrange, const uint4 &b,
                                                u32 *xs, u32 xn) {
    u64 d;
    const bool mem = inrange && bb_candidate(a, b, fwd, G, G5, d) && (d < bd || (d == bd && j < bj));
    const u32 m = __ballot_sync(0xFFFFFFFFu, mem);
    if (mem) {
        const u32 o = xn + __popc(m & lanemask_lt());
        if (o < FX_XCAP) xs[o] = j;
    }
    return xn + __popc(m);
}

// X(i) out of the search's own record: keep the entries that rank before the final pick (compacted in place)
__device__ __forceinline__ u32 fx_filter_seen(const uint4 *__restrict__ rec, const uint4 &a, bool fwd, u64 G, u64 G5, u64 bd, u32 bj, u32 *xs,
                                              u32 seen) {
    const u32 lane = lane_id();
    u32 out = 0;
    for (u32 q0 = 0; q0 < seen; q0 += 32) {
        const u32 q = q0 + lane;
        u32 j = NONE32;
        bool mem = false;
        if (q < seen) {
            j = xs[q];
            u64 d;
            mem = bb_candidate(a, rec[j], fwd, G, G5, d) && (d < bd || (d == bd && j < bj));
        }
        __syncwarp(); // the chunk is in registers before anything is written (out <= q0)
        const u32 m = __ballot_sync(0xFFFFFFFFu, mem);
        if (mem) xs[out + __popc(m & lanemask_lt())] = j;
        out += __popc(m);
        __syncwarp();
    }
    return out;
}

// One round of a bucket scan: the gap rule for every candidate of the round first (registers only), then the snapshot words of
// those that beat the best so far — independent gathers, one memory round trip — then the verdicts in order.  (Loading the
// words lazily, candidate by candidate, made a blocked candidate cost two dependent round trips; a position deep in a conflict
// meets dozens of them before its first eligible one.)
template <u32 CW>
__device__ __forceinline__ void fx_eval_round(const FxArrays &f, const uint4 &a, bool fwd, u64 G, u64 G5, const uint2 (&rb)[CW], const u32 (&rj)[CW],
                                              const bool (&in)[CW], u64 &bd, u32 &bj, const FxExtra &ex) {
    u64 dd[CW];
    bool want[CW];
    uint4 sn[CW];
#pragma unroll
    for (u32 k = 0; k < CW; k++) {
        want[k] = false;
        dd[k] = 0;
        if (in[k]) {
            const uint4 rec = make_uint4(rb[k].x, 0, rb[k].y, rb[k].y); // the gap rule reads query_start and t' only
            u64 d;
            if (bb_candidate(a, rec, fwd, G, G5, d) && (d < bd || (d == bd && rj[k] < bj))) { want[k] = true; dd[k] = d; }
        }
    }
#pragma unroll
    for (u32 k = 0; k < CW; k++)
        if (want[k]) sn[k] = f.snap[2 * (size_t)rj[k]];
    u64 ld = bd;
    u32 lj = bj;
#pragma unroll
    for (u32 k = 0; k < CW; k++)
        if (want[k] && (dd[k] < ld || (dd[k] == ld && rj[k] < lj))) {
            const u64 mp = ((u64)sn[k].y << 32) | sn[k].x;
            if (dd[k] < mp || ex.packed(rj[k], dd[k], sn[k].z, sn[k].w)) { ld = dd[k]; lj = rj[k]; }
        }
    bb_argmin(ld, lj);
    bd = ld;
    bj = lj;
}

// The search of k_fx_recompute over the target-bucket order.  The query-axis window of a position in a centromeric pile holds
// 10^5 candidates of which the target-gap rule admits a few dozen (configs[4]: the scattered half of the pile); in bucket order
// the candidates whose target coordinate can satisfy the rule (paf_filter.rs:812-833: target_start within [te - G/5, te + G] on
// the '+' strand, target_end within [ts - G, ts + G/5] on '-') are the entries of at most two buckets, and inside a bucket the
// entries are in position order, i.e. by query_start: the same pruned outward scans as bb_best_successor_warp run there, from
// the first entry whose query_start reaches query_end(i).  The arg-min is over (d, j) explicitly, so the reference's "first
// minimal j" does not depend on the visiting order, and every candidate ranking before the final pick is visited (pruning drops
// only candidates with q_gap^2 > best d), which is all the blocked-candidate record needs.
// COLLECT = false: bd / bj receive the pick.  COLLECT = true: bd / bj are the final pick; the valid candidates ranking before
// it are appended to xs (X(i)); returns their number.
template <bool COLLECT>
__device__ __forceinline__ u32 fx_bucket_pass(const FxArrays &f, u32 i, const uint4 &a, bool fwd, u64 G, u64 G5, u64 &bd, u32 &bj, FxExtra ex,
                                              u32 *xs) {
    const u32 full = 0xFFFFFFFFu;
    const u32 lane = lane_id();
    constexpr u32 CW = 4; // chunks per round
    u32 xn = 0;
    if (!COLLECT) { bd = NONE64; bj = NONE32; }
    // the candidate's target coordinate t' (start on '+', end on '-') against c: r_gap = |t' - c|, admitted down to c - below, up to c + above
    const u64 c = fwd ? a.w : a.z;
    const u64 below = fwd ? G5 : G, above = fwd ? G : G5;
    const u64 W = 1ull << f.bshift;
    const long long blo = (long long)((c > below ? c - below : 0) >> f.bshift), bhi = (long long)min((c + above) >> f.bshift, (u64)f.dirD - 2);
    const long long bc = (long long)(c >> f.bshift);
    const u32 *dir = f.dir + (size_t)f.hg[i] * f.dirD;
    // buckets outwards from the one that holds c: a bucket whose nearest edge is further than sqrt(best d) holds no better candidate
    bool live_up = true, live_dn = true; // buckets still worth a visit in either direction
    for (long long step = 0; live_up || live_dn; step++) {
        for (int side = 0; side < 2; side++) {
            if ((side && step == 0) || !(side ? live_dn : live_up)) continue;
            const long long b = side ? bc - step : bc + step;
            if (b < blo || b > bhi) { (side ? live_dn : live_up) = false; continue; }
            const u64 rmin = step == 0 ? 0 : (side ? c - ((u64)(b + 1) * W - 1) : (u64)b * W - c);
            const u64 r2 = rmin * rmin; // every candidate of the bucket has d >= q_gap^2 + r2
            if (r2 > bd) { (side ? live_dn : live_up) = false; continue; } // and every bucket beyond it
            const u32 lo0 = dir[b], hi0 = dir[b + 1];
            if (lo0 == hi0) continue;
            // first entry of the bucket whose query_start reaches query_end(i): 33-ary search, 32 probes in flight per round
            u32 lo = lo0, hi = hi0;
            while (hi - lo > 32) {
                const u32 width = hi - lo;
                const u32 p = lo + (u32)(((u64)(lane + 1) * width) / 33);
                const u32 nb = __popc(__ballot_sync(full, f.bq[p].x < a.y));
                const u32 nlo = nb ? lo + (u32)(((u64)nb * width) / 33) + 1 : lo;
                const u32 nhi = nb < 32 ? lo + (u32)(((u64)(nb + 1) * width) / 33) : hi;
                lo = nlo;
                hi = nhi;
            }
            if (hi > lo) {
                const u32 p = lo + lane;
                lo += __popc(__ballot_sync(full, p < hi && f.bq[p].x < a.y));
            }
            const u32 org = lo;
            for (u32 base = org; base < hi0; base += 32 * CW) { // right of the origin: q_gap = qs - qe >= 0 grows
                uint2 rb[CW];
                u32 rj[CW];
#pragma unroll
                for (u32 k = 0; k < CW; k++) {
                    const u32 m = base + k * 32 + lane;
                    rb[k] = make_uint2(0, 0);
                    rj[k] = NONE32;
                    if (m < hi0) { rb[k] = f.bq[m]; rj[k] = f.bk[m]; }
                }
                bool mono = false;
                bool in[CW];
#pragma unroll
                for (u32 k = 0; k < CW; k++) {
                    mono = false;
                    if (rj[k] != NONE32) {
                        const u64 qg = (u64)rb[k].x - a.y;
                        mono = qg <= G && qg * qg + r2 <= bd;
                    }
                    in[k] = mono && rj[k] > i; // (a zero-length record meets earlier positions with the same start here)
                }
                if (COLLECT) {
#pragma unroll
                    for (u32 k = 0; k < CW; k++)
                        xn = fx_collect_chunk(a, fwd, G, G5, bd, bj, rj[k], in[k], make_uint4(rb[k].x, 0, rb[k].y, rb[k].y), xs, xn);
                } else fx_eval_round<CW>(f, a, fwd, G, G5, rb, rj, in, bd, bj, ex);
                if (!__shfl_sync(full, (int)mono, 31)) break; // monotone: once the last candidate is out, so is everything further right
            }
            for (u32 top = org; top > lo0;) { // left of the origin: overlap = qe - qs > 0 grows going left, positions descend
                const u32 cnt = min(32u * CW, top - lo0);
                uint2 rb[CW];
                u32 rj[CW];
#pragma unroll
                for (u32 k = 0; k < CW; k++) {
                    const u32 off = k * 32 + lane;
                    rb[k] = make_uint2(0, 0);
                    rj[k] = NONE32;
                    if (off < cnt) { rb[k] = f.bq[top - 1 - off]; rj[k] = f.bk[top - 1 - off]; }
                }
                bool in[CW];
#pragma unroll
                for (u32 k = 0; k < CW; k++) {
                    in[k] = false;
                    if (rj[k] != NONE32) {
                        const u64 ov = (u64)a.y - rb[k].x;
                        in[k] = ov <= G5 && ov * ov + r2 <= bd && rj[k] > i;
                    }
                }
                if (COLLECT) {
#pragma unroll
                    for (u32 k = 0; k < CW; k++)
                        xn = fx_collect_chunk(a, fwd, G, G5, bd, bj, rj[k], in[k], make_uint4(rb[k].x, 0, rb[k].y, rb[k].y), xs, xn);
                } else fx_eval_round<CW>(f, a, fwd, G, G5, rb, rj, in, bd, bj, ex);
                if (cnt < 32 * CW || !__shfl_sync(full, (int)in[CW - 1], 31)) break;
                top -= 32 * CW;
            }
        }
    }
    return xn;
}

// step 3: one warp per listed position
__global__ void __launch_bounds__(128, 8) k_fx_recompute(FxArrays f, u64 G) {
    __shared__ u32 s_x[4][FX_XCAP];
    __shared__ u32 s_seen[4];
    const u32 full = 0xFFFFFFFFu;
    const u32 lane = lane_id();
    const u64 G5 = G / 5;
    u32 *xs = s_x[threadIdx.x >> 5];
    const u32 n_list = f.ctrs[0];
    while (true) {
        u32 w = 0;
        if (lane == 0) w = atomicAdd(&f.ctrs[2], 1u);
        w = __shfl_sync(full, w, 0);
        if (w >= n_list) break;
        const u32 i = f.list[w];
        const uint4 a = f.rec[i];
        const bool fwd = !(f.gend[i] & FX_REV);
        u64 bd;
        u32 bj;
        u32 *n_seen = &s_seen[threadIdx.x >> 5];
        if (lane == 0) *n_seen = 0;
        __syncwarp();
        FxExtra ex{f, i, xs, n_seen};
        fx_bucket_pass<false>(f, i, a, fwd, G, G5, bd, bj, ex, nullptr);
        __syncwarp();
        // X(i): normally out of the search's own record of blocked candidates; a separate pruned pass if that overflowed
        const u32 seen = *n_seen;
        const u32 xn = seen <= FX_XCAP && !f.force_collect ? fx_filter_seen(f.rec, a, fwd, G, G5, bd, bj, xs, seen)
                                                           : fx_bucket_pass<true>(f, i, a, fwd, G, G5, bd, bj, ex, xs);
        __syncwarp();
        u32 xo = 0;
        u16 xc = FX_XOVER;
        u32 hi = bj != NONE32 ? bj : i;
        if (xn <= FX_XCAP)
            for (u32 q = lane; q < xn; q += 32) hi = max(hi, xs[q]);
        hi = __reduce_max_sync(full, hi);
        if (lane == 0) {
            const u32 old = f.pick[i];
            if (bj != old) {
                atomicAdd(&f.ctrs[1], 1u);
                if (old != NONE32) f.dirty[old >> FX_DB] = 1; // the picker lists of both successors change
                if (bj != NONE32) f.dirty[bj >> FX_DB] = 1;
                if (old != NONE32) atomicOr(&f.dbits_w[old >> 5], 1u << (old & 31));
                if (bj != NONE32) atomicOr(&f.dbits_w[bj >> 5], 1u << (bj & 31));
            }
            f.xhi[i] = hi;
            f.pick[i] = bj;
            f.pd[i] = bd;
            if (xn <= FX_XCAP) {
                if (xn <= f.xcap[i]) { xo = f.xoff[i]; xc = (u16)xn; }
                else { // a new slot (the old one is abandoned): capacity rounded up to a power of two >= 4, so X(i) can grow in place
                    const u32 cap = xn <= 4 ? 4u : 1u << (32 - __clz(xn - 1));
                    const unsigned long long at = atomicAdd(f.pool_top, (unsigned long long)cap);
                    if (at + cap <= (unsigned long long)f.pool_cap) { xo = (u32)at; xc = (u16)xn; f.xoff[i] = xo; f.xcap[i] = (u16)cap; }
                    else atomicAdd(&f.ctrs[3], 1u);
                }
            }
            f.xcnt[i] = xc;
        }
        xo = __shfl_sync(full, xo, 0);
        xc = (u16)__shfl_sync(full, (u32)xc, 0);
        if (xc != FX_XOVER)
            for (u32 q = lane; q < xn; q += 32) {
                const u32 jx = xs[q];
                f.pool[xo + q] = jx;
                u64 d = 0;
                bb_candidate(a, f.rec[jx], fwd, G, G5, d); // valid by construction (fx_filter_seen / the collect pass)
                f.pool_d[xo + q] = d;
            }
        __syncwarp();
    }
}

// Resolve the huge groups.  hpos[k] = sorted position of k (ascending); gid / gstart / n_groups describe the groups in
// sorted-position space.  Writes root[] for the positions of huge groups and returns true; returns false (root[] untouched)
// if the picks have not settled after SWG_FIXPOINT_MAX_ROUNDS rounds (default 256): a dependency chain that long is walked
// faster sequentially, and the caller hands the groups to k_chain_resolve_warp.  The first round evaluates every position
// against an empty snapshot (that IS the unconstrained arg-min), all searches go through fx_bucket_pass.  maxcoord bounds
// every coordinate.
static bool chain_fixpoint(swg_ctx *c, u32 n_h, const u32 *hpos, const uint4 *srec, const u64 *skey, int cb, const u32 *gid, const u32 *gstart,
                           u32 n_groups, u32 n_m, u64 G, u32 *root, u32 *bsum, u32 maxcoord) {
    cudaStream_t st = c->stream;
    LaunchCounter &lc = c->lc;
    Arena &A = c->arena;
    const bool verbose = c->knobs.stage_timing;
    FxArrays f;
    f.n = n_h;
    f.rec = A.take<uint4>(n_h);
    f.gend = A.take<u32>(n_h);
    f.pick = A.take<u32>(n_h);
    f.pd = A.take<u64>(n_h);
    f.cnt = A.take<u32>(n_h);
    f.off = A.take<u32>((size_t)n_h + 1);
    f.minpi = A.take<u32>(n_h);
    f.firstp = A.take<u32>(n_h);
    f.li = nullptr; // the sorted positions of each round's sort
    f.force_collect = c->knobs.fx_force_collect;
    f.ld = A.take<u64>(n_h);
    f.xoff = A.take<u32>(n_h);
    f.xcnt = A.take<u16>(n_h);
    f.xcap = A.take<u16>(n_h);
    {   // X(i) pool: mean |X| grows with the density of the pile (about 9 on the '-' strand group of a 5 M pile, ten times
        // that at 50 M); slots are powers of two and an outgrown slot is abandoned, so be generous where memory allows
        size_t free_b = 0, total_b = 0;
        SWG_CUDA(cudaMemGetInfo(&free_b, &total_b));
        const u64 want = (u64)n_h * 96 + 4096, fit = free_b / 2 / 12;
        f.pool_cap = (u32)std::min<u64>(std::min<u64>(want, std::max<u64>(fit, (u64)n_h * 8 + 4096)), 0xF0000000ull);
    }
    f.pool = A.take<u32>(f.pool_cap);
    f.pool_d = A.take<u64>(f.pool_cap);
    f.pool_top = A.take<unsigned long long>(1);
    f.list = A.take<u32>(n_h);
    const u32 n_blk = (n_h >> FX_DB) + 1;
    f.xhi = A.take<u32>(n_h);
    f.dirty = A.take<u32>(n_blk);
    f.dps = A.take<u32>((size_t)n_blk + 1);
    f.use_dirty = 0;
    const size_t n_bw = ((size_t)n_h >> 5) + 1;
    f.dbits = A.take<u32>(n_bw);
    f.dbits_w = A.take<u32>(n_bw);
    f.ctrs = A.take<u32>(4);
    u32 *scan_tot = A.take<u32>(1);
    SWG_CUDA(cudaMemsetAsync(f.xcnt, 0, sizeof(u16) * (size_t)n_h, st));
    SWG_CUDA(cudaMemsetAsync(f.xcap, 0, sizeof(u16) * (size_t)n_h, st));
    SWG_CUDA(cudaMemsetAsync(f.pool_top, 0, sizeof(unsigned long long), st));
    {
        const FxArrays g = f;
        launch_for<t_fx_init>(n_h, st, lc, [=] __device__(u32 k) {
            const u32 p = hpos[k];
            const u32 gr = gid[p];
            const u32 e = (gr + 1 < n_groups) ? gstart[gr + 1] : n_m;
            const bool fwd = ((skey[p] >> cb) & 1) == 0;
            g.rec[k] = srec[p];
            g.gend[k] = (k + (e - p)) | (fwd ? 0u : FX_REV);
            g.pick[k] = NONE32;
            g.xhi[k] = k;
            g.pd[k] = NONE64;
        });
    }
    u32 *h = reinterpret_cast<u32 *>(c->h_ctr + C_COUNT);
    // dense numbers of the huge groups (a group starts where the previous position's group ends)
    f.hg = A.take<u32>(n_h);
    f.snap = A.take<uint4>(2 * (size_t)n_h);
    {
        const FxArrays g = f;
        scan_apply([=] __device__(u32 k) -> u32 { return (k == 0 || (g.gend[k - 1] & ~FX_REV) == k) ? 1u : 0u; },
                   [=] __device__(u32 k, u32 ex, u32 v) { g.hg[k] = ex + v - 1; }, n_h, bsum, scan_tot, st, lc);
    }
    SWG_CUDA(cudaMemcpyAsync(h, scan_tot, sizeof(u32), cudaMemcpyDeviceToHost, st));
    SWG_CUDA(cudaStreamSynchronize(st));
    const u32 n_hg = h[0];
    // bucket width: 1/32 of the smallest power of two >= G + G/5 + 1 (SWG_FX_BUCKET_NARROW=<log2 of the divisor>: tuning aid).
    // A search visits the buckets outwards from the one that holds its own target coordinate and stops at the first whose
    // nearest edge is further than sqrt(best d): narrow buckets keep the scans of the dense diagonal short, wide ones spare
    // the scattered positions origin searches.  Wider if the directory (one entry per group and bucket) would pass 2^25
    // entries or 2^20 per group.
    int bs = std::max(bits_for(G + G / 5) - c->knobs.fx_bucket_narrow, 4);
    while (((((u64)maxcoord >> bs) + 2) * n_hg > (1ull << 25) || ((u64)maxcoord >> bs) + 2 > (1ull << 20)) && bs < 32) bs++;
    f.bshift = bs;
    const u32 nbk = (u32)(((u64)maxcoord >> bs) + 1);
    f.dirD = nbk + 1;
    const int tb = bits_for(nbk - 1 ? nbk - 1 : 1);
    const size_t n_dir = (size_t)n_hg * f.dirD + 1;
    u64 *bkey = A.take<u64>(n_h), *bkey2 = A.take<u64>(n_h);
    u32 *bv = A.take<u32>(n_h), *bv2 = A.take<u32>(n_h);
    {
        const FxArrays g = f;
        launch_for<t_fx_bkey>(n_h, st, lc, [=] __device__(u32 k) {
            const uint4 r = g.rec[k];
            const u32 t = (g.gend[k] & FX_REV) ? r.w : r.z; // '-' strand: the rule tests the candidate's target_end
            bkey[k] = ((u64)g.hg[k] << tb) | ((u64)t >> bs);
            bv[k] = k;
        });
    }
    sort_pairs(c, bkey, bkey2, bv, bv2, n_h, tb + bits_for(n_hg > 1 ? n_hg - 1 : 1)); // stable: positions ascend inside a bucket
    f.bk = bv;
    f.bq = A.take<uint2>(n_h);
    f.dir = A.take<u32>(n_dir);
    {
        const FxArrays g = f;
        const u64 *ks = bkey;
        const u32 D = f.dirD;
        launch_for<t_fx_brec>(n_h, st, lc, [=] __device__(u32 m) {
            {
                const u32 k = g.bk[m];
                const uint4 r = g.rec[k];
                g.bq[m] = make_uint2(r.x, (g.gend[k] & FX_REV) ? r.w : r.z);
            }
            // directory: dir[x] = first entry whose (group, bucket) slot is >= x
            const u64 km = ks[m];
            const u64 slot = (km >> tb) * D + (km & ((1ull << tb) - 1));
            u64 from = 0;
            if (m > 0) { const u64 kp = ks[m - 1]; from = (kp >> tb) * D + (kp & ((1ull << tb) - 1)) + 1; }
            for (u64 x = from; x <= slot; x++) g.dir[x] = m;
            if (m + 1 == g.n)
                for (u64 x = slot + 1; x < n_dir; x++) g.dir[x] = g.n;
        });
    }
    if (verbose) fprintf(stderr, "[swg fixpoint] target buckets: %u huge groups, 2^%d wide, %u per group\n", n_hg, bs, nbk);
    int rounds = 0;
    u64 total_recomputed = 0;
    auto t_round = std::chrono::steady_clock::now();
    {
        // round 0: every position against the empty snapshot = the unconstrained arg-min (nothing is blocked: X(i) stays empty).
        // A thread scans the next successors of its position first; only a window that goes on is left to the warp search.
        SWG_CUDA(cudaMemsetAsync(f.minpi, 0xFF, sizeof(u32) * (size_t)n_h, st));
        SWG_CUDA(cudaMemsetAsync(f.firstp, 0xFF, sizeof(u32) * (size_t)n_h, st));
        SWG_CUDA(cudaMemsetAsync(f.off, 0, sizeof(u32) * ((size_t)n_h + 1), st));
        SWG_CUDA(cudaMemsetAsync(f.snap, 0xFF, 2 * sizeof(uint4) * (size_t)n_h, st)); // nobody picks anybody
        SWG_CUDA(cudaMemsetAsync(f.dbits_w, 0, sizeof(u32) * n_bw, st));
        SWG_CUDA(cudaMemsetAsync(f.dirty, 0, sizeof(u32) * (size_t)n_blk, st));
        SWG_CUDA(cudaMemsetAsync(f.ctrs, 0, 4 * sizeof(u32), st));
        k_fx_round0_linear<<<cdiv(n_h, 256), 256, 0, st>>>(f, G);
        k_fx_recompute<<<(u32)c->sm_count * 8, 128, 0, st>>>(f, G);
        lc.n += 2;
        if (verbose) {
            SWG_CUDA(cudaStreamSynchronize(st));
            const auto t1 = std::chrono::steady_clock::now();
            fprintf(stderr, "[swg fixpoint] round 0 (unconstrained picks, bucket order): %.2f ms\n", std::chrono::duration<double, std::milli>(t1 - t_round).count());
            t_round = t1;
        }
    }
    // picker lists in position order (stable sort of the positions by their pick), picker d as prefix minima
    u64 *sk = A.take<u64>(n_h), *sk2 = A.take<u64>(n_h);
    u32 *sv = A.take<u32>(n_h), *sv2 = A.take<u32>(n_h);
    const RadixSortPlan sp = rs_plan(n_h, 0, bits_for(n_h));
    void *stmp = A.take<char>(sp.temp_bytes);
    while (true) {
        {
            const FxArrays gs = f;
            u64 *kk = sk;
            u32 *vv = sv;
            launch_for<t_fx_skey>(n_h, st, lc, [=] __device__(u32 k) {
                const u32 j = gs.pick[k];
                kk[k] = j == NONE32 ? gs.n : j; // positions without a pick sort behind every list
                vv[k] = k;
            });
            rs_sort_pairs(sp, sk, sk2, sv, sv2, stmp, st, c->sm_count, lc);
            f.li = sv;
        }
        // 0. which blocks of successors saw a picker list change in the last round (prefix counts for k_fx_check_warp)
        if (rounds > 0) {
            const FxArrays gd = f;
            scan_apply([=] __device__(u32 b) -> u32 { return gd.dirty[b]; },
                       [=] __device__(u32 b, u32 ex, u32 v) {
                           gd.dps[b] = ex;
                           if (b + 1 == n_blk) gd.dps[n_blk] = ex + v;
                       },
                       n_blk, bsum, scan_tot, st, lc);
            f.use_dirty = 1;
        }
        SWG_CUDA(cudaMemsetAsync(f.dirty, 0, sizeof(u32) * (size_t)n_blk, st));
        // what the last round's re-evaluations marked is read by this round's check
        std::swap(f.dbits, f.dbits_w);
        SWG_CUDA(cudaMemsetAsync(f.dbits_w, 0, sizeof(u32) * n_bw, st));
        // 1. snapshot of the picks
        const FxArrays g = f;
        SWG_CUDA(cudaMemsetAsync(f.cnt, 0, sizeof(u32) * (size_t)n_h, st));
        SWG_CUDA(cudaMemsetAsync(f.ctrs, 0, 4 * sizeof(u32), st));
        launch_for<t_fx_count>(n_h, st, lc, [=] __device__(u32 k) {
            const u32 j = g.pick[k];
            if (j != NONE32) atomicAdd(&g.cnt[j], 1u);
        });
        scan_apply([=] __device__(u32 k) -> u32 { return g.cnt[k]; },
                   [=] __device__(u32 k, u32 ex, u32 v) {
                       g.off[k] = ex;
                       if (k + 1 == g.n) g.off[g.n] = ex + v;
                   },
                   n_h, bsum, scan_tot, st, lc);
        // one pass per successor over its list (position order): prefix minima, who holds the minimum first, the packed words
        launch_for<t_fx_pm>(n_h, st, lc, [=] __device__(u32 j) {
            const u32 a = g.off[j], b = g.off[j + 1];
            u64 m = NONE64, fd = NONE64;
            u32 mi = NONE32, fp = NONE32;
            for (u32 p = a; p < b; p++) {
                const u32 k = g.li[p];
                const u64 d = g.pd[k];
                if (p == a) { fp = k; fd = d; }
                if (d < m) { m = d; mi = k; }
                g.ld[p] = m;
            }
            g.minpi[j] = mi; g.firstp[j] = fp;
            g.snap[2 * (size_t)j] = make_uint4((u32)m, (u32)(m >> 32), mi, fp);
            g.snap[2 * (size_t)j + 1] = make_uint4((u32)fd, (u32)(fd >> 32), a, b - a);
        });
        // 2. + 3.
        double ms_snap = 0, ms_check = 0;
        auto lap = [&](double &ms) { // diagnostics only (SWG_STAGE_TIMING): where a round spends its time
            if (!verbose) return;
            SWG_CUDA(cudaStreamSynchronize(st));
            const auto t1 = std::chrono::steady_clock::now();
            ms = std::chrono::duration<double, std::milli>(t1 - t_round).count();
        };
        lap(ms_snap);
        k_fx_check_warp<<<cdiv(n_h, 256), 256, 0, st>>>(f, G);
        lap(ms_check);
        k_fx_recompute<<<(u32)c->sm_count * 8, 128, 0, st>>>(f, G);
        lc.n += 2;
        SWG_CUDA(cudaMemcpyAsync(h, f.ctrs, 4 * sizeof(u32), cudaMemcpyDeviceToHost, st));
        if (verbose) SWG_CUDA(cudaMemcpyAsync(h + 4, f.pool_top, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
        SWG_CUDA(cudaStreamSynchronize(st));
        rounds++;
        total_recomputed += h[0];
        if (verbose) {
            const auto t1 = std::chrono::steady_clock::now();
            fprintf(stderr, "[swg fixpoint] round %d: %u of %u positions re-evaluated, %u picks changed, %.2f ms (snapshot %.2f, check %.2f), pool %llu of %u (%u refused)\n", rounds,
                    h[0], n_h, h[1], std::chrono::duration<double, std::milli>(t1 - t_round).count(), ms_snap, ms_check - ms_snap,
                    (unsigned long long)(h[4] | ((u64)h[5] << 32)), f.pool_cap, h[3]);
            t_round = t1;
        }
        if (h[1] == 0) break; // the snapshot of this round equals the picks: it is the fixed point
        if (rounds >= c->knobs.fixpoint_max_rounds) {
            if (verbose) fprintf(stderr, "[swg fixpoint] not settled after %d rounds (%u picks still changing): sequential walk instead\n", rounds, h[1]);
            return false;
        }
    }
    if (c->knobs.fixpoint_verify) {
        // Self-check for sizes no oracle reaches: (*) has exactly one solution, so it suffices that EVERY position, evaluated
        // from scratch against the final snapshot, reproduces its pick (this bypasses the X(i) bookkeeping of k_fx_check_warp).
        const FxArrays g = f;
        SWG_CUDA(cudaMemsetAsync(f.ctrs, 0, 4 * sizeof(u32), st));
        launch_for<t_fx_all>(n_h, st, lc, [=] __device__(u32 k) {
            g.list[k] = k;
            if (k == 0) g.ctrs[0] = g.n;
        });
        k_fx_recompute<<<(u32)c->sm_count * 8, 128, 0, st>>>(f, G);
        lc.n++;
        SWG_CUDA(cudaMemcpyAsync(h, f.ctrs, 4 * sizeof(u32), cudaMemcpyDeviceToHost, st));
        SWG_CUDA(cudaStreamSynchronize(st));
        if (verbose) fprintf(stderr, "[swg fixpoint] verification: %u of %u positions would change their pick\n", h[1], n_h);
        if (h[1] != 0) throw RangeError{"fixed-point chaining: verification failed (" + std::to_string(h[1]) + " positions)"};
    }
    // pred[j] = the last picker of j; roots by pointer jumping (in place: a racing read sees an older or a newer
    // ancestor, both valid), bits_for(n) + 1 rounds cover any chain length
    {
        const FxArrays g = f;
        u32 *r = f.list;
        launch_for<t_fx_pred>(n_h, st, lc, [=] __device__(u32 j) {
            u32 m = NONE32;
            for (u32 p = g.off[j]; p < g.off[j + 1]; p++) m = (m == NONE32 || g.li[p] > m) ? g.li[p] : m;
            r[j] = m == NONE32 ? j : m;
        });
        for (int k = 0; k < bits_for(n_h) + 1; k++)
            launch_for<t_fx_jump>(n_h, st, lc, [=] __device__(u32 j) {
                const u32 a = r[j];
                const u32 b = r[a];
                if (b != a) r[j] = b;
            });
        launch_for<t_fx_scatter>(n_h, st, lc, [=] __device__(u32 k) { root[hpos[k]] = hpos[r[k]]; });
    }
    if (verbose) fprintf(stderr, "[swg fixpoint] %u positions in huge groups, %d rounds, %llu re-evaluations\n", n_h, rounds,
                         (unsigned long long)total_recomputed);
    return true;
}

} // namespace swg

// sweepga_oracle.cpp — CPU restatement of the sweepga mapping filter.
//
// TEST INFRASTRUCTURE, NOT PRODUCT.  Only tests/, __graft_entry__.smoke() and
// bench.py's cpu_baseline / --impl reference legs may load this library.  The
// product (sweepga_b200/csrc) never links, calls or falls back to it.
//
// Parity status: PINNED against the reference's own known-answer tests
// (tests/test_reference_vectors.py transcribes them with file:line), the Rust
// reference itself cannot be compiled here (no cargo/rustc, un-vendored deps).
// Exceptions: orc_ani_stats (the ANI pre-pass, src/main.rs:334-688) and
// orc_tree_filter_paf (src/tree_filter.rs:205-283) — PARITY UNPINNED: the reference
// holds no test or vector for them (beyond extract_genome_prefix); tests/test_host.py
// and tests/test_tree_cpu.py check the restatements against answers computed by hand
// from the source, and the SipHash-1-3 core against CPython's siphash13.
//
// Every function cites the reference file:line it restates
// (paths relative to /root/reference).  Containers: BTreeSet -> std::set with
// the same comparator, IndexMap/IndexSet -> insertion-ordered map (IndexMap
// below), HashSet iteration at paf_filter.rs:638 -> canonicalised (see
// rescue()).  Arithmetic: u64 integers, f64, glibc log/sqrt — as the reference.
//
// Build: g++ -O2 -std=c++17 -shared -fPIC -o liboracle.so sweepga_oracle.cpp
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <map>
#include <set>
#include <string>
#include <unordered_map>
#include <unordered_set>
#include <vector>

#include "../include/sweepga_b200.h" // swg_config POD + enum values only

namespace orc {

static const uint64_t USIZE_MAX = ~(uint64_t)0;

// Insertion-ordered map (indexmap::IndexMap): iteration = first-insertion order.
template <class K, class V, class H = std::hash<K>> struct IndexMap {
    std::unordered_map<K, size_t, H> pos;
    std::vector<std::pair<K, V>> items;
    V &entry(const K &k) {
        auto it = pos.find(k);
        if (it == pos.end()) {
            pos.emplace(k, items.size());
            items.emplace_back(k, V());
            return items.back().second;
        }
        return items[it->second].second;
    }
};
struct PairHash {
    size_t operator()(const std::pair<uint64_t, uint64_t> &p) const {
        return std::hash<uint64_t>()(p.first * 0x9E3779B97F4A7C15ull ^ (p.second + 0x7F4A7C15ull + (p.first << 6)));
    }
};
typedef std::pair<uint64_t, uint64_t> Key2;

// ---------------------------------------------------------------------------
// plane_sweep_exact.rs
// ---------------------------------------------------------------------------
struct PSM { // PlaneSweepMapping, plane_sweep_exact.rs:10-18
    uint64_t qs, qe, ts, te;
    double identity;
    bool discard, overlapped;
};

// score_with_function, plane_sweep_exact.rs:29-86 (length = query span on BOTH axes)
static double score_of(const PSM &m, int scoring) {
    double length = (double)(uint64_t)(m.qe - m.qs);
    switch (scoring) {
    case SWG_SCORE_IDENTITY:
        return (m.identity <= 0.0) ? -INFINITY : m.identity;
    case SWG_SCORE_LENGTH:
        return (length <= 0.0) ? -INFINITY : length;
    case SWG_SCORE_LENGTH_IDENTITY:
    case SWG_SCORE_MATCHES:
        return (length <= 0.0 || m.identity <= 0.0) ? -INFINITY : length * m.identity;
    default: // LogLengthIdentity
        return (length <= 0.0 || m.identity <= 0.0) ? -INFINITY : m.identity * std::log(length);
    }
}

// query_overlap / target_overlap, plane_sweep_exact.rs:113-144
static double overlap_frac(uint64_t s1, uint64_t e1, uint64_t s2, uint64_t e2) {
    uint64_t os = std::max(s1, s2), oe = std::min(e1, e2);
    int64_t d = (int64_t)oe - (int64_t)os;
    double overlap_len = (double)(d > 0 ? d : 0);
    double l1 = (double)(uint64_t)(e1 - s1), l2 = (double)(uint64_t)(e2 - s2);
    double min_len = std::min(l1, l2);
    return (min_len > 0.0) ? overlap_len / min_len : 0.0;
}

struct MappingOrder { // plane_sweep_exact.rs:163-194
    size_t idx;
    double score;
    uint64_t start_pos;
};
struct MappingOrderLess {
    bool operator()(const MappingOrder &a, const MappingOrder &b) const {
        // other.score.partial_cmp(self.score).unwrap_or(Equal): score DESC, NaN compares Equal
        if (a.score > b.score) return true;
        if (a.score < b.score) return false;
        if (a.start_pos != b.start_pos) return a.start_pos < b.start_pos;
        return a.idx < b.idx;
    }
};
typedef std::set<MappingOrder, MappingOrderLess> Bst;

// mark_good, plane_sweep_exact.rs:197-259
static void mark_good(const Bst &bst, std::vector<PSM> &m, uint64_t to_keep, double thr, int axis,
                      std::vector<size_t> &kept_indices, std::vector<uint8_t> &in_kept) {
    if (bst.empty()) return;
    kept_indices.clear();
    uint64_t kept = 0;
    for (auto it = bst.begin(); it != bst.end(); ++it, ++kept) {
        if (kept >= to_keep) break;
        m[it->idx].discard = false;
        kept_indices.push_back(it->idx);
    }
    if (thr < 1.0) {
        for (size_t k : kept_indices) in_kept[k] = 1; // the reference's per-call HashSet
        for (auto it = bst.begin(); it != bst.end(); ++it) {
            size_t idx = it->idx;
            if (in_kept[idx]) continue;
            for (size_t k : kept_indices) {
                double ov = (axis == 0) ? overlap_frac(m[idx].qs, m[idx].qe, m[k].qs, m[k].qe)
                                        : overlap_frac(m[idx].ts, m[idx].te, m[k].ts, m[k].te);
                if (ov > thr) {
                    m[idx].overlapped = true;
                    m[idx].discard = true;
                    break;
                }
            }
        }
        for (size_t k : kept_indices) in_kept[k] = 0;
    }
}

// plane_sweep_query / plane_sweep_target, plane_sweep_exact.rs:268-433 (axis 0 = query, 1 = target)
static std::vector<size_t> plane_sweep_axis(std::vector<PSM> &m, uint64_t to_keep, double thr, int scoring, int axis) {
    std::vector<size_t> out;
    if (m.size() <= 1) {
        for (size_t i = 0; i < m.size(); i++) out.push_back(i);
        return out;
    }
    for (auto &x : m) { x.discard = true; x.overlapped = false; }
    struct Event { uint64_t pos; int type; size_t idx; };
    std::vector<Event> ev;
    ev.reserve(m.size() * 2);
    for (size_t i = 0; i < m.size(); i++) {
        ev.push_back({axis == 0 ? m[i].qs : m[i].ts, 0, i});
        ev.push_back({axis == 0 ? m[i].qe : m[i].te, 1, i});
    }
    std::stable_sort(ev.begin(), ev.end(), [](const Event &a, const Event &b) {
        if (a.pos != b.pos) return a.pos < b.pos;
        return a.type < b.type;
    });
    Bst bst;
    std::vector<size_t> kept_indices;
    std::vector<uint8_t> in_kept(m.size(), 0);
    size_t i = 0;
    while (i < ev.size()) {
        uint64_t cur = ev[i].pos;
        size_t j = i;
        while (j < ev.size() && ev[j].pos == cur) j++;
        for (size_t e = i; e < j; e++) {
            size_t k = ev[e].idx;
            MappingOrder mo{k, score_of(m[k], scoring), axis == 0 ? m[k].qs : m[k].ts};
            if (ev[e].type == 0) bst.insert(mo); else bst.erase(mo);
        }
        mark_good(bst, m, to_keep, thr, axis, kept_indices, in_kept);
        i = j;
    }
    for (size_t k = 0; k < m.size(); k++)
        if (!m[k].discard && !m[k].overlapped) out.push_back(k);
    return out;
}

// plane_sweep_both, plane_sweep_exact.rs:436-461 (query sweep, then target sweep over the survivors)
static std::vector<size_t> plane_sweep_both(std::vector<PSM> &m, uint64_t nq, uint64_t nt, double thr, int scoring) {
    std::vector<size_t> qk = plane_sweep_axis(m, nq, thr, scoring, 0);
    std::vector<PSM> f;
    f.reserve(qk.size());
    for (size_t i : qk) f.push_back(m[i]);
    std::vector<size_t> tk = plane_sweep_axis(f, nt, thr, scoring, 1);
    std::vector<size_t> out;
    out.reserve(tk.size());
    for (size_t i : tk) out.push_back(qk[i]);
    return out;
}

// ---------------------------------------------------------------------------
// plane_sweep_core.rs:80-201 (secondary API; different semantics on purpose)
// ---------------------------------------------------------------------------
struct Interval { uint32_t begin, end; double score; };
static bool core_overlaps(const Interval &a, const Interval &b, double thr) { // :20-33
    uint32_t os = std::max(a.begin, b.begin), oe = std::min(a.end, b.end);
    if (os >= oe) return false;
    uint32_t ol = oe - os;
    uint32_t ml = std::min(a.end - a.begin, b.end - b.begin);
    return (double)ol / (double)ml > thr;
}
static std::vector<size_t> plane_sweep_core(const std::vector<Interval> &iv, uint64_t max_keep, double thr) {
    std::vector<size_t> kept;
    if (iv.empty()) return kept;
    if (iv.size() == 1) { kept.push_back(0); return kept; }
    if (max_keep == USIZE_MAX) { for (size_t i = 0; i < iv.size(); i++) kept.push_back(i); return kept; }
    struct Ev { uint32_t pos; int type; size_t idx; };
    std::vector<Ev> ev;
    for (size_t i = 0; i < iv.size(); i++) { ev.push_back({iv[i].begin, 0, i}); ev.push_back({iv[i].end, 1, i}); }
    // sort_unstable on (pos, Begin<End): ties between equal (pos,type) are processed in an
    // unspecified order, but insertion/removal of a set commute, and mark_best only runs after
    // each Begin: the kept SET can depend on the order of equal Begins.  We use stable order.
    std::stable_sort(ev.begin(), ev.end(), [](const Ev &a, const Ev &b) {
        if (a.pos != b.pos) return a.pos < b.pos;
        return a.type < b.type;
    });
    std::set<std::pair<int64_t, size_t>> active; // (-score_bits as i64, idx)
    for (auto &e : ev) {
        uint64_t bits;
        std::memcpy(&bits, &iv[e.idx].score, 8);
        int64_t key = -(int64_t)bits;
        if (e.type == 0) {
            active.insert({key, e.idx});
            uint64_t c = 0;
            for (auto it = active.begin(); it != active.end() && c < max_keep; ++it, ++c) kept.push_back(it->second);
        } else {
            active.erase({key, e.idx});
        }
    }
    std::sort(kept.begin(), kept.end());
    kept.erase(std::unique(kept.begin(), kept.end()), kept.end());
    if (thr < 1.0 && kept.size() > 1) { // filter_by_overlap :167-201
        std::stable_sort(kept.begin(), kept.end(), [&](size_t a, size_t b) { return iv[a].score > iv[b].score; });
        std::vector<size_t> fin{kept[0]};
        for (size_t t = 1; t < kept.size(); t++) {
            bool keep = true;
            for (size_t k : fin)
                if (core_overlaps(iv[kept[t]], iv[k], thr)) { keep = false; break; }
            if (keep) fin.push_back(kept[t]);
        }
        kept = fin;
    }
    return kept;
}

// ---------------------------------------------------------------------------
// union_find.rs:3-64
// ---------------------------------------------------------------------------
struct UnionFind {
    std::vector<size_t> parent, rank;
    explicit UnionFind(size_t n) : parent(n), rank(n, 0) { for (size_t i = 0; i < n; i++) parent[i] = i; }
    size_t find(size_t x) {
        size_t r = x;
        while (parent[r] != r) r = parent[r];
        while (parent[x] != r) { size_t nx = parent[x]; parent[x] = r; x = nx; } // path compression
        return r;
    }
    void unite(size_t x, size_t y) {
        size_t rx = find(x), ry = find(y);
        if (rx == ry) return;
        if (rank[rx] < rank[ry]) parent[rx] = ry;
        else if (rank[rx] > rank[ry]) parent[ry] = rx;
        else { parent[ry] = rx; rank[rx]++; }
    }
    std::vector<std::vector<size_t>> get_sets() { // ascending root, members ascending
        std::map<size_t, std::vector<size_t>> g;
        for (size_t i = 0; i < parent.size(); i++) g[find(i)].push_back(i);
        std::vector<std::vector<size_t>> out;
        for (auto &kv : g) out.push_back(std::move(kv.second));
        return out;
    }
};

// ---------------------------------------------------------------------------
// paf_filter.rs
// ---------------------------------------------------------------------------
struct Rec { // RecordMeta, paf_filter.rs:52-71 (names interned to ids)
    size_t rank; // here: index into the caller's table
    uint32_t qid, tid;
    uint64_t qs, qe, ts, te, blen, matches;
    double identity;
    bool fwd;
};
struct Chain { // MergedChain, paf_filter.rs:142-155
    uint32_t qid, tid;
    uint64_t qs, qe, ts, te;
    bool fwd;
    uint64_t total_length;
    double weighted_identity;
    uint64_t sum_matches, sum_block;
    std::vector<size_t> members; // ranks
    size_t B = 0;                // first member (in M order) of the chain's (q,t,strand) group: its first-appearance key
};

struct Tables {
    const uint32_t *P, *P2;
};

// apply_plane_sweep_to_mappings, paf_filter.rs:972-1123
static std::vector<Rec> primary_sweep(const std::vector<Rec> &mappings, const swg_config &cfg, const Tables &tb) {
    if (mappings.size() <= 1) return mappings;
    uint64_t qlim, tlim;
    switch (cfg.mapping_filter_mode) { // :1004-1014
    case SWG_ONE_TO_ONE: qlim = 1; tlim = 1; break;
    case SWG_ONE_TO_MANY:
        qlim = cfg.mapping_max_per_query != SWG_NO_LIMIT ? cfg.mapping_max_per_query : 1;
        tlim = cfg.mapping_max_per_target; // None -> usize::MAX (same encoding)
        break;
    default:
        qlim = cfg.mapping_max_per_query;
        tlim = cfg.mapping_max_per_target;
    }
    IndexMap<Key2, std::vector<size_t>, PairHash> genome_pairs; // :1037-1046
    for (size_t i = 0; i < mappings.size(); i++)
        genome_pairs.entry({tb.P[mappings[i].qid], tb.P[mappings[i].tid]}).push_back(i);

    std::vector<size_t> all_kept;
    std::vector<uint8_t> qkept(mappings.size(), 0), tkept(mappings.size(), 0);
    for (auto &gp : genome_pairs.items) {
        const std::vector<size_t> &gidx = gp.second;
        for (int axis = 0; axis < 2; axis++) { // :1055-1100
            IndexMap<uint64_t, std::vector<size_t>> by_seq;
            for (size_t idx : gidx) by_seq.entry(axis == 0 ? mappings[idx].qid : mappings[idx].tid).push_back(idx);
            for (auto &grp : by_seq.items) {
                const std::vector<size_t> &ind = grp.second;
                std::vector<PSM> pm;
                pm.reserve(ind.size());
                for (size_t i : ind) pm.push_back({mappings[i].qs, mappings[i].qe, mappings[i].ts, mappings[i].te, mappings[i].identity, false, false});
                std::vector<size_t> kept = plane_sweep_axis(pm, axis == 0 ? qlim : tlim, cfg.overlap_threshold, cfg.scoring_function, axis);
                for (size_t k : kept) (axis == 0 ? qkept : tkept)[ind[k]] = 1;
            }
        }
        for (size_t idx : gidx) // intersection, ascending (:1105-1111)
            if (qkept[idx] && tkept[idx]) all_kept.push_back(idx);
    }
    std::vector<Rec> out;
    out.reserve(all_kept.size());
    for (size_t i : all_kept) out.push_back(mappings[i]);
    return out;
}

struct Key3Hash {
    size_t operator()(const std::pair<Key2, int> &k) const { return PairHash()(k.first) * 31 + k.second; }
};

// merge_mappings_into_chains, paf_filter.rs:750-933
static std::vector<Chain> merge_into_chains(const std::vector<Rec> &md, uint64_t max_gap) {
    IndexMap<std::pair<Key2, int>, std::vector<size_t>, Key3Hash> groups; // :761-770
    for (size_t i = 0; i < md.size(); i++) groups.entry({{md[i].qid, md[i].tid}, md[i].fwd ? 1 : 0}).push_back(i);
    std::vector<Chain> all;
    for (auto &g : groups.items) {
        bool fwd = g.first.second == 1;
        std::vector<size_t> s = g.second;
        std::stable_sort(s.begin(), s.end(), [&](size_t a, size_t b) { return md[a].qs < md[b].qs; }); // :776-777
        size_t n = s.size();
        std::vector<uint64_t> bps(n, ~(uint64_t)0);
        std::vector<int64_t> bpi(n, -1);
        for (size_t i = 0; i < n; i++) { // :784-851
            const Rec &a = md[s[i]];
            uint64_t bound = a.qe + max_gap;
            int64_t best_j = -1;
            uint64_t best = ~(uint64_t)0;
            for (size_t j = i + 1; j < n; j++) {
                const Rec &b = md[s[j]];
                if (b.qs > bound) break;
                uint64_t qgap;
                if (b.qs >= a.qe) qgap = b.qs - a.qe;
                else { uint64_t ov = a.qe - b.qs; qgap = (ov <= max_gap / 5) ? ov : max_gap + 1; }
                uint64_t rgap;
                if (fwd) {
                    if (b.ts >= a.te) rgap = b.ts - a.te;
                    else { uint64_t ov = a.te - b.ts; rgap = (ov <= max_gap / 5) ? ov : max_gap + 1; }
                } else if (a.ts >= b.te) rgap = a.ts - b.te;
                else { uint64_t ov = b.te - a.ts; rgap = (ov <= max_gap / 5) ? ov : max_gap + 1; }
                if (qgap <= max_gap && rgap <= max_gap) {
                    uint64_t d = qgap * qgap + rgap * rgap;
                    if (d < best && d < bps[j]) { best = d; best_j = (int64_t)j; }
                }
            }
            if (best_j >= 0) { bps[best_j] = best; bpi[best_j] = (int64_t)i; }
        }
        UnionFind uf(n); // :854-866
        for (size_t j = 0; j < n; j++) if (bpi[j] >= 0) uf.unite((size_t)bpi[j], j);
        for (auto &set : uf.get_sets()) {
            if (set.empty()) continue;
            Chain c;
            c.B = md[g.second[0]].rank;
            c.qid = (uint32_t)g.first.first.first; c.tid = (uint32_t)g.first.first.second; c.fwd = fwd;
            uint64_t qmin = ~(uint64_t)0, qmax = 0, tmin = ~(uint64_t)0, tmax = 0, sm = 0, sb = 0;
            for (size_t k : set) { // :875-894
                const Rec &r = md[s[k]];
                qmin = std::min(qmin, r.qs); qmax = std::max(qmax, r.qe);
                tmin = std::min(tmin, r.ts); tmax = std::max(tmax, r.te);
                c.members.push_back(r.rank);
                sm += r.matches; sb += r.blen;
            }
            uint64_t total = qmax - qmin;
            uint64_t gap = total > sb ? total - sb : 0; // saturating_sub
            double lg = gap > 0 ? std::max(std::log((double)gap), 0.0) : 0.0;
            double eff = (double)sb + lg;
            c.qs = qmin; c.qe = qmax; c.ts = tmin; c.te = tmax;
            c.total_length = total; c.sum_matches = sm; c.sum_block = sb;
            c.weighted_identity = eff > 0.0 ? (double)sm / eff : 0.0;
            all.push_back(std::move(c));
        }
    }
    return all;
}

// apply_scaffold_plane_sweep + plane_sweep_scaffolds, paf_filter.rs:1126-1146, plane_sweep_scaffold.rs:47-251
static std::vector<size_t> scaffold_sweep(const std::vector<Chain> &chains, const swg_config &cfg, const Tables &tb) {
    std::vector<size_t> all;
    if (chains.size() <= 1) { for (size_t i = 0; i < chains.size(); i++) all.push_back(i); return all; }
    uint64_t nq, nt;
    if (cfg.scaffold_filter_mode == SWG_ONE_TO_ONE) { nq = 1; nt = 1; }
    else {
        nq = cfg.scaffold_max_per_query; // None -> usize::MAX (same encoding)
        nt = cfg.scaffold_max_per_target;
    }
    IndexMap<Key2, IndexMap<Key2, std::vector<size_t>, PairHash>, PairHash> gp;
    for (size_t i = 0; i < chains.size(); i++)
        gp.entry({tb.P2[chains[i].qid], tb.P2[chains[i].tid]}).entry({chains[i].qid, chains[i].tid}).push_back(i);
    for (auto &g : gp.items)
        for (auto &cp : g.second.items) {
            const std::vector<size_t> &ind = cp.second;
            std::vector<PSM> pm;
            for (size_t i : ind) pm.push_back({chains[i].qs, chains[i].qe, chains[i].ts, chains[i].te, chains[i].weighted_identity, false, false});
            for (size_t k : plane_sweep_both(pm, nq, nt, cfg.scaffold_overlap_threshold, cfg.scoring_function)) all.push_back(ind[k]);
        }
    return all;
}

struct Stats { uint64_t v[10]; };

// apply_filters, paf_filter.rs:379-747.  status/chain are indexed like the input table.
static void apply_filters(const std::vector<Rec> &input, const swg_config &cfg, const Tables &tb,
                          uint8_t *status, uint32_t *chain_out, swg_stats *st, uint32_t *keyA = nullptr, uint32_t *keyB = nullptr) {
    size_t n_in = input.size();
    for (size_t i = 0; i < n_in; i++) { status[i] = SWG_DROPPED; chain_out[i] = 0; }
    std::vector<Rec> md; // :384-388
    for (const Rec &m : input)
        if (m.blen >= cfg.min_block_length && (cfg.keep_self || m.qid != m.tid) && m.identity >= cfg.min_identity) md.push_back(m);
    std::vector<Rec> all_orig = md; // :391
    if (st) { st->n_input = n_in; st->n_stage1 = md.size(); }
    md = primary_sweep(md, cfg, tb); // :400
    if (st) st->n_after_sweep = md.size();
    if (cfg.scaffold_gap == 0) { // :409-434
        for (const Rec &m : md) status[m.rank] = SWG_UNASSIGNED;
        if (st) st->n_kept = md.size();
        return;
    }
    std::vector<Chain> merged = merge_into_chains(md, cfg.scaffold_gap); // :441
    if (st) st->n_chains = merged.size();
    std::vector<Chain> filtered; // :449-455
    for (Chain &c : merged)
        if (c.total_length >= cfg.min_scaffold_length && c.weighted_identity >= cfg.min_scaffold_identity) filtered.push_back(std::move(c));
    if (st) st->n_chains_after_mass = filtered.size();
    std::unordered_set<size_t> pre_members; // :471-476
    for (const Chain &c : filtered) for (size_t r : c.members) pre_members.insert(r);
    {
        std::vector<size_t> kept = scaffold_sweep(filtered, cfg, tb); // :478
        if (keyA && keyB) {
            // merge keys for multi-shard numbering (not part of the reference): per kept chain, the first-appearance
            // indices (A: genome pair over the stage-1 records, B: group over M) of the first filtered chain of its
            // genome-pair group (plane_sweep_scaffold.rs:116-130 iteration order)
            std::unordered_map<Key2, size_t, PairHash> firstA;
            for (const Rec &m : all_orig) firstA.emplace(Key2{tb.P[m.qid], tb.P[m.tid]}, m.rank);
            std::unordered_map<Key2, size_t, PairHash> g2first;
            for (size_t i = 0; i < filtered.size(); i++) g2first.emplace(Key2{tb.P2[filtered[i].qid], tb.P2[filtered[i].tid]}, i);
            for (size_t k = 0; k < kept.size(); k++) {
                const Chain &f = filtered[g2first[Key2{tb.P2[filtered[kept[k]].qid], tb.P2[filtered[kept[k]].tid]}]];
                keyA[k] = (uint32_t)firstA[Key2{tb.P[f.qid], tb.P[f.tid]}];
                keyB[k] = (uint32_t)f.B;
            }
        }
        std::vector<Chain> k2;
        for (size_t i : kept) k2.push_back(filtered[i]);
        filtered.swap(k2);
    }
    if (st) st->n_chains_kept = filtered.size();
    if (cfg.scaffolds_only) { // :486-513
        uint64_t nk = 0;
        for (size_t ci = 0; ci < filtered.size(); ci++)
            for (size_t r : filtered[ci].members) { status[r] = SWG_SCAFFOLD; chain_out[r] = (uint32_t)(ci + 1); nk++; }
        if (st) { st->n_kept = nk; st->n_anchors = nk; }
        return;
    }
    std::unordered_map<size_t, uint32_t> anchor_chain; // anchor_ranks + rank_to_chain_id, :517-528
    for (size_t ci = 0; ci < filtered.size(); ci++)
        for (size_t r : filtered[ci].members) anchor_chain[r] = (uint32_t)(ci + 1);
    // inversion capture, :535-597
    uint64_t G = cfg.scaffold_gap;
    std::unordered_map<Key2, std::vector<size_t>, PairHash> rev_by_pair;
    for (size_t i = 0; i < all_orig.size(); i++)
        if (!all_orig[i].fwd) rev_by_pair[{all_orig[i].qid, all_orig[i].tid}].push_back(i);
    for (size_t ci = 0; ci < filtered.size(); ci++) {
        const Chain &c = filtered[ci];
        if (!c.fwd) continue;
        int64_t diag = (int64_t)c.ts - (int64_t)c.qs;
        auto it = rev_by_pair.find({c.qid, c.tid});
        if (it == rev_by_pair.end()) continue;
        for (size_t idx : it->second) {
            const Rec &m = all_orig[idx];
            if (anchor_chain.count(m.rank)) continue;
            uint64_t ext_s = c.qs > G ? c.qs - G : 0;                          // saturating_sub
            uint64_t ext_e = (c.qe + G < c.qe) ? ~(uint64_t)0 : c.qe + G;      // saturating_add
            if (m.qe < ext_s || m.qs > ext_e) continue;
            uint64_t qc = (m.qs + m.qe) / 2, tc = (m.ts + m.te) / 2;
            int64_t dv = (int64_t)tc - (int64_t)qc - diag;
            uint64_t dev = dv < 0 ? (uint64_t)(-dv) : (uint64_t)dv;
            uint64_t perp = (uint64_t)((double)dev / M_SQRT2);
            if (perp <= G) anchor_chain[m.rank] = (uint32_t)(ci + 1);
        }
    }
    // lost = pre_sweep_scaffold_members - anchors, :601-604
    // rescue, :613-747
    IndexMap<Key2, std::vector<size_t>, PairHash> by_pair;
    for (size_t i = 0; i < all_orig.size(); i++) by_pair.entry({all_orig[i].qid, all_orig[i].tid}).push_back(i);
    std::unordered_map<Key2, std::vector<size_t>, PairHash> anchors_by_pair;
    for (size_t i = 0; i < all_orig.size(); i++)
        if (anchor_chain.count(all_orig[i].rank)) anchors_by_pair[{all_orig[i].qid, all_orig[i].tid}].push_back(i);
    uint64_t D = cfg.scaffold_max_deviation, n_resc = 0, n_kept = 0;
    for (auto &pr : by_pair.items) {
        auto ait = anchors_by_pair.find(pr.first);
        if (ait == anchors_by_pair.end() || ait->second.empty()) continue; // :658-660
        const std::vector<size_t> &anch = ait->second;
        for (size_t mi : pr.second) {
            const Rec &m = all_orig[mi];
            auto ac = anchor_chain.find(m.rank);
            if (ac != anchor_chain.end()) { status[m.rank] = SWG_SCAFFOLD; chain_out[m.rank] = ac->second; n_kept++; continue; }
            if (pre_members.count(m.rank)) continue; // member of a swept-away scaffold: never rescued
            if (D == 0) continue;
            uint64_t qc = (m.qs + m.qe) / 2, tc = (m.ts + m.te) / 2;
            // The reference takes the first anchor (HashSet iteration order — nondeterministic,
            // paf_filter.rs:638-643,690-716) whose distance is <= D.  Membership in the result is
            // order-independent; the chain id is canonicalised here as: smallest distance, then
            // smallest anchor index.
            uint64_t best_d = ~(uint64_t)0; size_t best_a = 0; bool found = false;
            for (size_t ai : anch) {
                const Rec &a = all_orig[ai];
                uint64_t aqc = (a.qs + a.qe) / 2;
                int64_t qd_ = (int64_t)qc - (int64_t)aqc;
                uint64_t qd = qd_ < 0 ? (uint64_t)(-qd_) : (uint64_t)qd_;
                if (qd > D) continue;
                uint64_t atc = (a.ts + a.te) / 2;
                int64_t td_ = (int64_t)tc - (int64_t)atc;
                uint64_t td = td_ < 0 ? (uint64_t)(-td_) : (uint64_t)td_;
                uint64_t dist = (uint64_t)std::sqrt((double)(qd * qd + td * td));
                if (dist <= D && (!found || dist < best_d || (dist == best_d && a.rank < best_a))) { best_d = dist; best_a = a.rank; found = true; }
            }
            if (found) { status[m.rank] = SWG_RESCUED; chain_out[m.rank] = anchor_chain[best_a]; n_resc++; n_kept++; }
        }
    }
    if (st) { st->n_anchors = anchor_chain.size(); st->n_rescued = n_resc; st->n_kept = n_kept; }
}

// ---------------------------------------------------------------------------
// extract_metadata, paf_filter.rs:292-376; parse_cigar_counts, paf.rs:32-64
// ---------------------------------------------------------------------------
static bool rust_parse_u64(const std::string &s, uint64_t &out) { // str::parse::<u64>
    size_t i = 0;
    if (s.empty()) return false;
    if (s[0] == '+') i = 1;
    if (i >= s.size()) return false;
    uint64_t v = 0;
    for (; i < s.size(); i++) {
        if (s[i] < '0' || s[i] > '9') return false;
        uint64_t d = (uint64_t)(s[i] - '0');
        if (v > (~(uint64_t)0 - d) / 10) return false;
        v = v * 10 + d;
    }
    out = v;
    return true;
}
static bool rust_parse_f64(const std::string &s, double &out) { // str::parse::<f64> (decimal grammar, inf/nan)
    if (s.empty()) return false;
    for (char c : s) if (c == 'x' || c == 'X' || c == ' ' || c == '\t' || c == 'p' || c == 'P' || c == '(') return false;
    const char *b = s.c_str();
    char *e = nullptr;
    double v = strtod(b, &e);
    if (e != b + s.size()) return false;
    out = v;
    return true;
}
static bool cigar_matches(const std::string &cg, uint64_t &matches) {
    uint64_t m = 0;
    std::string num;
    for (char ch : cg) {
        if (ch >= '0' && ch <= '9') num.push_back(ch);
        else {
            uint64_t c;
            if (!rust_parse_u64(num, c)) return false; // Err => tag ignored
            num.clear();
            if (ch == '=') m += c;
        }
    }
    matches = m;
    return true;
}

struct Paf {
    std::vector<uint64_t> rank, qs, qe, ts, te, blen, matches;
    std::vector<uint32_t> qid, tid;
    std::vector<double> identity;
    std::vector<uint8_t> strand;
    std::vector<std::string> names;
    std::vector<uint32_t> P, P2;
    std::vector<std::string> lines; // every input line (for the writer)
};

static uint32_t intern(std::unordered_map<std::string, uint32_t> &m, const std::string &s) {
    auto it = m.find(s);
    if (it != m.end()) return it->second;
    uint32_t id = (uint32_t)m.size();
    m.emplace(s, id);
    return id;
}
static std::string prefix_P(const std::string &n) { // paf_filter.rs:1022-1030
    size_t p = n.rfind('#');
    return p == std::string::npos ? n : n.substr(0, p + 1);
}
static std::string prefix_P2(const std::string &n) { // plane_sweep_scaffold.rs:13-22
    size_t p = n.find('#');
    if (p == std::string::npos) return n;
    size_t p2 = n.find('#', p + 1);
    std::string f1 = (p2 == std::string::npos) ? n.substr(p + 1) : n.substr(p + 1, p2 - p - 1);
    return n.substr(0, p) + "#" + f1 + "#";
}

static Paf *parse_paf(const char *path) {
    std::ifstream in(path, std::ios::binary);
    if (!in) return nullptr;
    Paf *p = new Paf();
    std::unordered_map<std::string, uint32_t> name_id, p_id, p2_id;
    std::string line;
    uint64_t rank = 0;
    while (std::getline(in, line)) { // BufRead::lines(): strips "\n" and a preceding "\r"
        if (!line.empty() && line.back() == '\r') line.pop_back();
        p->lines.push_back(line);
        std::vector<std::string> f;
        size_t s = 0;
        while (true) {
            size_t t = line.find('\t', s);
            if (t == std::string::npos) { f.push_back(line.substr(s)); break; }
            f.push_back(line.substr(s, t - s));
            s = t + 1;
        }
        uint64_t this_rank = rank++;
        if (f.size() < 11) continue; // :302-304 (still consumes a rank)
        auto u = [&](const std::string &x, uint64_t dflt) { uint64_t v; return rust_parse_u64(x, v) ? v : dflt; };
        uint64_t qs = u(f[2], 0), qe = u(f[3], 0), ts = u(f[7], 0), te = u(f[8], 0), mt = u(f[9], 0), bl = u(f[10], 1);
        double identity = (double)mt / (double)std::max<uint64_t>(bl, 1);
        uint64_t exact = mt;
        for (size_t k = 11; k < f.size(); k++) { // :326-343, in line order, later tag wins
            if (f[k].compare(0, 5, "dv:f:") == 0) {
                double dv;
                if (rust_parse_f64(f[k].substr(5), dv)) identity = 1.0 - dv;
            } else if (f[k].compare(0, 5, "cg:Z:") == 0) {
                uint64_t cm;
                if (cigar_matches(f[k].substr(5), cm) && cm > 0) { exact = cm; identity = (double)cm / (double)std::max<uint64_t>(bl, 1); }
            }
        }
        uint32_t qi = intern(name_id, f[0]);
        if (qi == p->names.size()) { p->names.push_back(f[0]); p->P.push_back(intern(p_id, prefix_P(f[0]))); p->P2.push_back(intern(p2_id, prefix_P2(f[0]))); }
        uint32_t ti = intern(name_id, f[5]);
        if (ti == p->names.size()) { p->names.push_back(f[5]); p->P.push_back(intern(p_id, prefix_P(f[5]))); p->P2.push_back(intern(p2_id, prefix_P2(f[5]))); }
        p->rank.push_back(this_rank); p->qid.push_back(qi); p->tid.push_back(ti);
        p->qs.push_back(qs); p->qe.push_back(qe); p->ts.push_back(ts); p->te.push_back(te);
        p->blen.push_back(bl); p->matches.push_back(exact); p->identity.push_back(identity);
        p->strand.push_back(f[4] == "+" ? '+' : '-');
    }
    return p;
}

} // namespace orc

// ---------------------------------------------------------------------------
// C entry points (ctypes)
// ---------------------------------------------------------------------------
extern "C" {

int orc_apply_filters(const swg_config *cfg, uint64_t n, const uint32_t *qid, const uint32_t *tid,
                      const uint64_t *qs, const uint64_t *qe, const uint64_t *ts, const uint64_t *te,
                      const uint64_t *blen, const uint64_t *matches, const double *identity,
                      const uint8_t *strand, const uint32_t *seq_P, const uint32_t *seq_P2,
                      uint8_t *status, uint32_t *chain_id, swg_stats *stats, uint32_t *chain_keyA, uint32_t *chain_keyB) {
    std::vector<orc::Rec> in(n);
    for (uint64_t i = 0; i < n; i++)
        in[i] = {(size_t)i, qid[i], tid[i], qs[i], qe[i], ts[i], te[i], blen[i], matches[i], identity[i], strand[i] == '+'};
    orc::Tables tb{seq_P, seq_P2};
    swg_stats local;
    std::memset(&local, 0, sizeof local);
    orc::apply_filters(in, *cfg, tb, status, chain_id, &local, chain_keyA, chain_keyB);
    if (stats) *stats = local;
    return 0;
}

// axis: 0 query, 1 target, 2 both (n_keep = query limit, n_keep2 = target limit)
int orc_plane_sweep(int axis, uint64_t n, const uint64_t *qs, const uint64_t *qe, const uint64_t *ts,
                    const uint64_t *te, const double *identity, uint64_t n_keep, uint64_t n_keep2,
                    double thr, int scoring, uint8_t *keep) {
    std::vector<orc::PSM> m(n);
    for (uint64_t i = 0; i < n; i++) m[i] = {qs[i], qe[i], ts[i], te[i], identity[i], false, false};
    std::vector<size_t> k = axis == 2 ? orc::plane_sweep_both(m, n_keep, n_keep2, thr, scoring)
                                      : orc::plane_sweep_axis(m, n_keep, thr, scoring, axis);
    for (uint64_t i = 0; i < n; i++) keep[i] = 0;
    for (size_t i : k) keep[i] = 1;
    return (int)k.size();
}

double orc_score(uint64_t qs, uint64_t qe, double identity, int scoring) {
    orc::PSM m{qs, qe, 0, 0, identity, false, false};
    return orc::score_of(m, scoring);
}

// score_with_function (plane_sweep_exact.rs:29-86) over columns
void orc_score_column(uint64_t n, const uint32_t *qs, const uint32_t *qe, const double *identity, int scoring, double *out) {
    for (uint64_t i = 0; i < n; i++) out[i] = orc_score(qs[i], qe[i], identity[i], scoring);
}
// weighted_identity of a chain from its aggregates (paf_filter.rs:896-913), the statement sequence of merge_chains above
void orc_chain_identity(uint64_t n, const uint64_t *total_length, const uint64_t *sum_block, const uint64_t *sum_matches, double *out) {
    for (uint64_t i = 0; i < n; i++) {
        const uint64_t total = total_length[i], sb = sum_block[i], sm = sum_matches[i];
        uint64_t gap = total > sb ? total - sb : 0; // saturating_sub
        double lg = gap > 0 ? std::max(std::log((double)gap), 0.0) : 0.0;
        double eff = (double)sb + lg;
        out[i] = eff > 0.0 ? (double)sm / eff : 0.0;
    }
}

// returns the number kept; out_idx receives the kept indices in the reference's output order
int orc_plane_sweep_core(uint64_t n, const uint32_t *begin, const uint32_t *end, const double *score,
                         uint64_t max_keep, double thr, uint64_t *out_idx) {
    std::vector<orc::Interval> iv(n);
    for (uint64_t i = 0; i < n; i++) iv[i] = {begin[i], end[i], score[i]};
    std::vector<size_t> k = orc::plane_sweep_core(iv, max_keep, thr);
    for (size_t i = 0; i < k.size(); i++) out_idx[i] = k[i];
    return (int)k.size();
}

void *orc_paf_parse(const char *path) { return orc::parse_paf(path); }
void orc_paf_free(void *h) { delete (orc::Paf *)h; }
uint64_t orc_paf_n(void *h) { return ((orc::Paf *)h)->rank.size(); }
uint64_t orc_paf_n_lines(void *h) { return ((orc::Paf *)h)->lines.size(); }
uint32_t orc_paf_n_seq(void *h) { return (uint32_t)((orc::Paf *)h)->names.size(); }
const char *orc_paf_seq_name(void *h, uint32_t i) { return ((orc::Paf *)h)->names[i].c_str(); }
// which: 0 rank 1 qs 2 qe 3 ts 4 te 5 blen 6 matches
const uint64_t *orc_paf_u64(void *h, int which) {
    orc::Paf *p = (orc::Paf *)h;
    switch (which) {
    case 0: return p->rank.data(); case 1: return p->qs.data(); case 2: return p->qe.data();
    case 3: return p->ts.data(); case 4: return p->te.data(); case 5: return p->blen.data();
    default: return p->matches.data();
    }
}
// which: 0 qid 1 tid 2 seq_P 3 seq_P2
const uint32_t *orc_paf_u32(void *h, int which) {
    orc::Paf *p = (orc::Paf *)h;
    switch (which) { case 0: return p->qid.data(); case 1: return p->tid.data(); case 2: return p->P.data(); default: return p->P2.data(); }
}
const double *orc_paf_identity(void *h) { return ((orc::Paf *)h)->identity.data(); }
const uint8_t *orc_paf_strand(void *h) { return ((orc::Paf *)h)->strand.data(); }

// write_filtered_output, paf_filter.rs:1689-1726.  status/chain indexed by RECORD (not line).
int orc_paf_write(void *h, const char *out_path, const uint8_t *status, const uint32_t *chain_id) {
    orc::Paf *p = (orc::Paf *)h;
    FILE *f = fopen(out_path, "wb");
    if (!f) return -1;
    size_t r = 0;
    static const char *names[4] = {"", "scaffold", "rescued", "unassigned"};
    for (size_t ln = 0; ln < p->lines.size(); ln++) {
        if (r < p->rank.size() && p->rank[r] == ln) {
            if (status[r] != SWG_DROPPED) {
                fputs(p->lines[ln].c_str(), f);
                if (chain_id[r]) fprintf(f, "\tch:Z:chain_%u", chain_id[r]);
                fprintf(f, "\tst:Z:%s\n", names[status[r]]);
            }
            r++;
        }
    }
    fclose(f);
    return 0;
}

// PafFilter::filter_paf restated end to end (parse + filter + write), for the CPU baseline.
int orc_filter_paf(const swg_config *cfg, const char *in_path, const char *out_path, swg_stats *stats) {
    orc::Paf *p = orc::parse_paf(in_path);
    if (!p) return -1;
    size_t n = p->rank.size();
    std::vector<uint8_t> status(n);
    std::vector<uint32_t> chain(n);
    orc_apply_filters(cfg, n, p->qid.data(), p->tid.data(), p->qs.data(), p->qe.data(), p->ts.data(), p->te.data(),
                      p->blen.data(), p->matches.data(), p->identity.data(), p->strand.data(), p->P.data(), p->P2.data(),
                      status.data(), chain.data(), stats, nullptr, nullptr);
    int rc = orc_paf_write(p, out_path, status.data(), chain.data());
    delete p;
    return rc;
}

// SipHash-1-3 with a zero key over g1 || 0xFF || g2 || 0xFF: std's DefaultHasher::new() fed `str::hash` twice
// (tree_filter.rs:147-151).  Restated from the SipHash specification; checked against CPython's siphash13 in tests/.
uint64_t orc_siphash13(const uint8_t *msg, uint64_t len) {
    auto rotl = [](uint64_t x, int b) { return (x << b) | (x >> (64 - b)); };
    uint64_t v0 = 0x736f6d6570736575ull, v1 = 0x646f72616e646f6dull, v2 = 0x6c7967656e657261ull, v3 = 0x7465646279746573ull; // k0 = k1 = 0
    auto round = [&]() {
        v0 += v1; v1 = rotl(v1, 13); v1 ^= v0; v0 = rotl(v0, 32);
        v2 += v3; v3 = rotl(v3, 16); v3 ^= v2;
        v0 += v3; v3 = rotl(v3, 21); v3 ^= v0;
        v2 += v1; v1 = rotl(v1, 17); v1 ^= v2; v2 = rotl(v2, 32);
    };
    uint64_t i = 0;
    for (; i + 8 <= len; i += 8) {
        uint64_t m = 0;
        for (int k = 0; k < 8; k++) m |= (uint64_t)msg[i + k] << (8 * k);
        v3 ^= m; round(); v0 ^= m;
    }
    uint64_t b = len << 56;
    for (int k = 0; i + k < len; k++) b |= (uint64_t)msg[i + k] << (8 * k);
    v3 ^= b; round(); v0 ^= b;
    v2 ^= 0xff;
    round(); round(); round();
    return v0 ^ v1 ^ v2 ^ v3;
}

// apply_tree_filter_to_paf, src/tree_filter.rs:205-283 (build_identity_matrix :39-80, select_tree_pairs :84-164,
// filter_tree_based :168-201).  The reference orders a genome's neighbours with a stable sort over HashMap iteration
// order, so ties in identity are broken arbitrarily there; here (and in the product) ties go by neighbour name.
// PARITY UNPINNED: the reference only tests extract_genome_prefix (tree_filter.rs:446-452).
int orc_tree_filter_paf(const char *in_path, const char *out_path, uint64_t k_nearest, uint64_t k_farthest, double random_fraction,
                        uint64_t *n_kept, uint64_t *n_selected) {
    using namespace orc;
    std::ifstream in(in_path, std::ios::binary);
    if (!in) return -1;
    struct Aln { std::string qg, tg; uint64_t m, b; };
    std::vector<Aln> alns;
    std::vector<std::string> lines;
    std::string line;
    while (std::getline(in, line)) {
        if (!line.empty() && line.back() == '\r') line.pop_back();
        if (line.empty() || line[0] == '#') continue; // :221-223
        std::vector<std::string> f;
        size_t s = 0;
        while (true) {
            size_t t = line.find('\t', s);
            if (t == std::string::npos) { f.push_back(line.substr(s)); break; }
            f.push_back(line.substr(s, t - s));
            s = t + 1;
        }
        if (f.size() < 11) continue;
        uint64_t m = 0, b = 1;
        if (!rust_parse_u64(f[9], m)) m = 0;
        if (!rust_parse_u64(f[10], b)) b = 1;
        alns.push_back(Aln{prefix_P2(f[0]), prefix_P2(f[5]), m, b}); // extract_genome_prefix :15-25 == the P2 rule
        lines.push_back(line);
    }
    std::map<std::pair<std::string, std::string>, std::pair<double, double>> sums; // :39-80
    for (const auto &a : alns) {
        if (a.qg == a.tg) continue;
        auto key = a.qg < a.tg ? std::make_pair(a.qg, a.tg) : std::make_pair(a.tg, a.qg);
        auto &e = sums[key];
        e.first += (double)a.m;
        e.second += (double)a.b;
    }
    std::map<std::pair<std::string, std::string>, double> ident;
    std::map<std::string, std::vector<std::pair<std::string, double>>> nb;
    for (const auto &kv : sums) {
        const double id = kv.second.second > 0.0 ? kv.second.first / kv.second.second : 0.0;
        ident[kv.first] = id;
        nb[kv.first.first].push_back({kv.first.second, id});
        nb[kv.first.second].push_back({kv.first.first, id});
    }
    std::set<std::pair<std::string, std::string>> selected; // :84-164
    for (auto &g : nb) {
        auto &v = g.second;
        for (auto &x : v) if (x.second != x.second) return -2; // partial_cmp().unwrap() panics on NaN
        std::sort(v.begin(), v.end(), [](const auto &x, const auto &y) { return x.second != y.second ? x.second > y.second : x.first < y.first; });
        auto add = [&](const std::string &o) { selected.insert(g.first < o ? std::make_pair(g.first, o) : std::make_pair(o, g.first)); };
        for (size_t k = 0; k < v.size() && k < k_nearest; k++) add(v[k].first);
        for (size_t k = 0; k < v.size() && k < k_farthest; k++) add(v[v.size() - 1 - k].first);
    }
    if (random_fraction > 0.0) {
        const double t = random_fraction * 18446744073709551615.0;
        const uint64_t thr = t >= 18446744073709551615.0 ? ~(uint64_t)0 : (t > 0.0 ? (uint64_t)t : 0); // `as u64` saturates
        for (const auto &kv : ident) {
            std::string msg = kv.first.first + "\xff" + kv.first.second + "\xff";
            if (orc_siphash13((const uint8_t *)msg.data(), msg.size()) <= thr) selected.insert(kv.first);
        }
    }
    FILE *out = fopen(out_path, "wb");
    if (!out) return -1;
    uint64_t kept = 0;
    for (size_t i = 0; i < alns.size(); i++) { // :168-201
        const auto &a = alns[i];
        if (a.qg == a.tg) continue;
        auto key = a.qg < a.tg ? std::make_pair(a.qg, a.tg) : std::make_pair(a.tg, a.qg);
        if (!selected.count(key)) continue;
        fwrite(lines[i].data(), 1, lines[i].size(), out);
        fputc('\n', out);
        kept++;
    }
    fclose(out);
    if (n_kept) *n_kept = kept;
    if (n_selected) *n_selected = selected.size();
    return 0;
}

// calculate_ani_stats + calculate_ani_n_percentile, src/main.rs:334-688.
// method 0 = All, 1 = Orthogonal (1:1 filter first, :346-383), 2 = NPercentile(percentile, sort); sort 0 = length,
// 1 = identity, 2 = score.  Returns 0 and *ani50; -1: I/O; -2: the reference would panic (NaN in partial_cmp).
int orc_ani_stats(const char *path, int method, double percentile, int sort, double *ani50, uint64_t *n_pairs) {
    using namespace orc;
    std::string input = path;
    std::string tmp;
    if (method == 1) { // :346-383
        swg_config c;
        memset(&c, 0, sizeof c);
        c.min_block_length = 1000;
        c.mapping_filter_mode = SWG_ONE_TO_ONE; c.mapping_max_per_query = 1; c.mapping_max_per_target = 1;
        c.scaffold_filter_mode = SWG_ONE_TO_ONE; c.scaffold_max_per_query = 1; c.scaffold_max_per_target = 1;
        c.overlap_threshold = 0.95; c.scaffold_gap = 10000; c.min_scaffold_length = 0; c.scaffold_overlap_threshold = 0.95;
        c.scaffold_max_deviation = 0; c.scoring_function = SWG_SCORE_MATCHES; c.min_identity = 0.0; c.min_scaffold_identity = 0.0;
        tmp = std::string(path) + ".orc_ani_tmp";
        if (orc_filter_paf(&c, path, tmp.c_str(), nullptr) != 0) return -1;
        input = tmp;
    }
    struct Aln { std::string qg, tg; double matches, block, identity; };
    std::vector<Aln> alns;
    std::unordered_map<std::string, uint64_t> genome_sizes;
    {
        std::ifstream in(input, std::ios::binary);
        if (!in) return -1;
        std::string line;
        while (std::getline(in, line)) {
            if (!line.empty() && line.back() == '\r') line.pop_back();
            if (line.empty() || line[0] == '#') continue; // :414-416 / :540-542
            std::vector<std::string> f;
            size_t s = 0;
            while (true) {
                size_t t = line.find('\t', s);
                if (t == std::string::npos) { f.push_back(line.substr(s)); break; }
                f.push_back(line.substr(s, t - s));
                s = t + 1;
            }
            if (f.size() < 11) continue;
            std::string qg = prefix_P(f[0]), tg = prefix_P(f[5]); // :424-433: up to and including the last '#'
            if (qg == tg) continue;                               // :436-438
            if (method == 2) {                                    // :560-575: sizes keyed by genome + last '#' field
                uint64_t ql = 0, tl = 0;
                if (!rust_parse_u64(f[1], ql)) ql = 0;
                if (!rust_parse_u64(f[6], tl)) tl = 0;
                auto last = [](const std::string &n) { size_t p = n.rfind('#'); return p == std::string::npos ? n : n.substr(p + 1); };
                genome_sizes.emplace(qg + last(f[0]), ql); // or_insert
                genome_sizes.emplace(tg + last(f[5]), tl);
            }
            double m = 0.0, b = 1.0;
            if (!rust_parse_f64(f[9], m)) m = 0.0;
            if (!rust_parse_f64(f[10], b)) b = 1.0;
            double fm = m;
            for (size_t k = 11; k < f.size(); k++) // :445-453: the FIRST dv:f: tag that parses
                if (f[k].compare(0, 5, "dv:f:") == 0) {
                    double dv;
                    if (rust_parse_f64(f[k].substr(5), dv)) { fm = (1.0 - dv) * b; break; }
                }
            // Rust's f64::max returns the other argument when one is NaN (std::max would return the NaN), so fmax
            alns.push_back(Aln{qg, tg, fm, b, fm / std::fmax(b, 1.0)});
        }
    }
    if (!tmp.empty()) remove(tmp.c_str());
    if (n_pairs) *n_pairs = 0;
    if (alns.empty()) { *ani50 = 0.0; return 0; } // :468-471 / :606-609
    size_t take = alns.size();
    if (method == 2) {
        // f64::max again (fmax): ln of a zero, negative or NaN block length is -inf or NaN, and the key then uses 1
        auto key = [&](const Aln &a) { return sort == 0 ? a.block : sort == 1 ? a.identity : a.identity * std::fmax(std::log(a.block), 1.0); };
        for (const auto &a : alns)
            if (key(a) != key(a)) return -2;
        std::stable_sort(alns.begin(), alns.end(), [&](const Aln &x, const Aln &y) { return key(x) > key(y); }); // :612-631
        double total = 0.0;
        for (const auto &kv : genome_sizes) total += (double)kv.second; // :634
        const double thr = total * (percentile / 100.0);                 // :638
        double cum = 0.0;
        take = 0;
        for (const auto &a : alns) { // :654-672: the alignment that crosses the threshold is still counted
            cum += a.block;
            take++;
            if (cum >= thr) break;
        }
    }
    std::map<std::pair<std::string, std::string>, std::pair<double, double>> pairs;
    for (size_t i = 0; i < take; i++) {
        const Aln &a = alns[i];
        auto key = a.qg < a.tg ? std::make_pair(a.qg, a.tg) : std::make_pair(a.tg, a.qg); // :455-459
        auto &e = pairs[key];
        e.first += a.matches;
        e.second += a.block;
    }
    std::vector<double> ani;
    for (const auto &kv : pairs) ani.push_back(kv.second.second > 0.0 ? kv.second.first / kv.second.second : 0.0);
    for (double v : ani) if (v != v) return -2;
    std::sort(ani.begin(), ani.end());
    const size_t mid = ani.size() / 2;
    *ani50 = (ani.size() % 2 == 0 && ani.size() > 1) ? (ani[mid - 1] + ani[mid]) / 2.0 : ani[mid]; // :490-495
    if (n_pairs) *n_pairs = ani.size();
    return 0;
}

} // extern "C"

// ani_device.cuh — the ANI pre-pass that sits in front of the filter (`--min-identity aniN`), on the device.
// (SURVEY §8f rank 4.)
//
//   ani_device  <- calculate_ani_stats + calculate_ani_n_percentile   (src/main.rs:334-688)
//
// The result is the median over genome pairs of  Σ matches / Σ block_length.  The reference accumulates both sums in
// f64, alignment by alignment — in file order (method "all") or in the order of a stable descending sort by block
// length / identity / score (method "nX"), cut where the cumulative block length reaches X % of the genome size.
// With dv:f: tags the addends are not integers, so the order of the additions is part of the result.  Here:
//   1. the text is tokenised on the device (k_ani_parse, built from the line grammar of paf_device.cuh; the lines it
//      lists are patched by the host reader through patch_lines, records compacted by take_records, names interned as
//      in the filter front end: ani_records)
//   2. "nX": one stable radix sort on the order-preserving bit pattern of the f64 key; the cut is found from per-tile
//      integer sums (exact while the block lengths are integers, which a PAF column always is; otherwise the host
//      walks the sorted column)
//   3. a second stable sort by genome pair brings every pair's addends together IN ORDER; one thread per pair adds them
//      sequentially (__dadd_rn, no reassociation), so the sums are the reference's bit for bit
//   4. the per-pair ANI values (a few thousand) go back; the host sorts them and takes the median.
#pragma once

namespace swg {

struct t_ani_pairs; struct t_ani_first; struct t_ani_sizes; struct t_ani_keys; struct t_ani_gather; struct t_ani_tiles;

struct AniPatch { u32 line; u32 kind; double m, b; u64 ql, tl; };

// One thread per line.  MODE 0: the ANI reader (main.rs:412-460 / :538-604): columns 2 / 7 as u64 into ql / tl, columns
// 10 / 11 as f64, the first dv:f: tag that parses.  MODE 1: the tree-filter reader (tree_filter.rs:219-245): columns
// 10 / 11 as u64 (unwrap_or 0 / 1) into ql / tl, no tags; the line length is kept for the output.  Both skip empty and
// '#' lines; the longest line is measured before the '\r' is stripped.
template <int MODE>
__global__ void __launch_bounds__(256) k_ani_parse(const char *__restrict__ text, const u64 *__restrict__ line_start, u32 n_lines, TokCols L,
                                                   u32 *__restrict__ fix_list, u64 *__restrict__ tc) {
    const u32 l = blockIdx.x * blockDim.x + threadIdx.x;
    bool ok = false;
    if (l < n_lines) {
        const u64 s = line_start[l];
        const char *line = text + s;
        const u32 len = strip_cr(line, line_len_raw(line_start, l));
        u8 kind = TK_SKIP;
        if (len > 0 && line[0] != '#') {
            u32 a = 0;
            bool fix = false, enough = true;
            u64 qh = 0, th = 0, ql = 0, tl = 0;
            u32 qlen = 0, trel = 0, tlen = 0;
            double m = 0.0, b = 1.0;
#pragma unroll 1
            for (int nf = 0; nf < 11; nf++) {
                u32 e = a;
                if (nf == 0 || nf == 5) {
                    const u64 hh = name_field(line, a, e, len);
                    if (nf == 0) { qh = hh; qlen = e - a; }
                    else { th = hh; trel = a; tlen = e - a; }
                } else if (MODE == 0 ? (nf == 1 || nf == 6) : (nf == 9 || nf == 10)) { // parse::<u64>().unwrap_or(0 | 1)
                    const u64 v = u64_field(line, a, e, len, (MODE == 1 && nf == 10) ? 1 : 0, fix);
                    if (nf == 1 || nf == 9) ql = v; else tl = v;
                } else {
                    while (e < len && line[e] != '\t') e++;
                    if (MODE == 0 && (nf == 9 || nf == 10)) { // parse::<f64>().unwrap_or(0.0 / 1.0)
                        double v;
                        const int rc = tok_parse_f64(line + a, e - a, v);
                        if (rc == 2) fix = true;
                        else if (rc == 1) { if (nf == 9) m = v; else b = v; }
                    }
                }
                if (e >= len) {
                    if (nf < 10) enough = false;
                    a = len + 1;
                    break;
                }
                a = e + 1;
            }
            if (enough) {
                double fm = m;
                if (MODE == 1) L.len[l] = len;
                while (MODE == 0 && a <= len && !fix) { // the first dv:f: tag that parses
                    u32 e = a;
                    while (e < len && line[e] != '\t') e++;
                    if (e - a >= 5 && line[a] == 'd' && line[a + 1] == 'v' && line[a + 2] == ':' && line[a + 3] == 'f' && line[a + 4] == ':') {
                        double dv;
                        const int rc = tok_parse_f64(line + a + 5, e - a - 5, dv);
                        if (rc == 1) { fm = __dmul_rn(__dsub_rn(1.0, dv), b); break; }
                        if (rc == 2) fix = true;
                    }
                    if (e >= len) break;
                    a = e + 1;
                }
                L.off[l] = s;
                L.qh[l] = qh; L.th[l] = th;
                L.qlen[l] = qlen; L.trel[l] = trel; L.tlen[l] = tlen;
                if (MODE == 0) { L.m[l] = fm; L.b[l] = b; }
                L.ql[l] = ql; L.tl[l] = tl;
                if (fix) {
                    kind = TK_FIX;
                    fix_list[atomicAdd((unsigned long long *)&tc[TC_NFIX], 1ull)] = l;
                } else kind = TK_OK;
            }
        }
        L.kind[l] = kind;
        ok = kind == TK_OK;
    }
    count_records(ok, tc);
    // the longest line sizes the output window of write_device (MODE 1); lines of 256 MiB and more are declined
    raise_maxlen(l < n_lines ? line_len_raw(line_start, l) : 0, tc);
}

// one thread per genome pair: the pair's addends are contiguous and in the reference's order
__global__ void __launch_bounds__(128) k_ani_pair_sums(const double *__restrict__ ms, const double *__restrict__ bs, const u32 *__restrict__ seg_start,
                                                       u32 n_pairs, u32 n_items, double *__restrict__ ani) {
    const u32 p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_pairs) return;
    const u32 s = seg_start[p], e = p + 1 < n_pairs ? seg_start[p + 1] : n_items;
    double sm = 0.0, sb = 0.0;
    u32 k = s;
    for (; k + 4 <= e; k += 4) { // independent loads first, then the dependent adds in order
        const double m0 = ms[k], m1 = ms[k + 1], m2 = ms[k + 2], m3 = ms[k + 3];
        const double b0 = bs[k], b1 = bs[k + 1], b2 = bs[k + 2], b3 = bs[k + 3];
        sm = __dadd_rn(__dadd_rn(__dadd_rn(__dadd_rn(sm, m0), m1), m2), m3);
        sb = __dadd_rn(__dadd_rn(__dadd_rn(__dadd_rn(sb, b0), b1), b2), b3);
    }
    for (; k < e; k++) { sm = __dadd_rn(sm, ms[k]); sb = __dadd_rn(sb, bs[k]); }
    ani[p] = sb > 0.0 ? __ddiv_rn(sm, sb) : 0.0; // main.rs:476-482
}

struct AniResult { double ani50 = 0.0; u64 n_pairs = 0; u64 n_alignments = 0; };
struct NanError {};

// The host readers of the lines k_ani_parse lists, as patch records.
static bool ani_reparse(const char *line, size_t len, AniPatch &p) {
    AniLine al;
    const bool ok = paf_ani_line(line, len, &al);
    p.kind = ok ? TK_OK : TK_SKIP; p.m = al.matches; p.b = al.block; p.ql = al.qlen; p.tl = al.tlen;
    return ok;
}
static bool tree_reparse(const char *line, size_t len, AniPatch &p) {
    AniLine al;
    p.ql = 0; p.tl = 1;
    const bool ok = paf_tree_line(line, len, &al, &p.ql, &p.tl);
    p.kind = ok ? TK_OK : TK_SKIP;
    return ok;
}

// The records of the ANI (MODE 0) or tree (MODE 1) reader: k_ani_parse, the host reader for the lines it lists, the
// compaction, and the names interned (*nt).  tc: the zeroed TC_COUNT counter block.  Returns 0 records (nothing else
// is set) when no line is an alignment.
template <int MODE>
static u32 ani_records(swg_ctx *c, const PafText &tx, const DevLines &dl, u64 *tc, TokCols *R, NameTable *nt) {
    constexpr u32 READER = MODE == 0 ? RD_ANI : RD_TREE;
    const TokCols L = take_cols<READER>(c->io, dl.n_lines);
    u32 *fix_list = c->io.take<u32>(dl.n_lines);
    u64 h_tc[TC_COUNT];
    k_ani_parse<MODE><<<cdiv(dl.n_lines, 256), 256, 0, c->stream>>>(dl.text, dl.line_start, dl.n_lines, L, fix_list, tc);
    c->lc.n++;
    tok_read(c, tc, h_tc);
    if (h_tc[TC_MAXLEN] > ((u64)256 << 20)) throw FrontEndFallback{"a line longer than 256 MiB"};
    c->tok_maxlen = (u32)h_tc[TC_MAXLEN];
    u64 n_ok = h_tc[TC_OK];
    if (h_tc[TC_NFIX]) // numbers outside the plain grammar: the host's line reader decides
        n_ok += patch_lines<AniPatch>(
            c, tx, dl, fix_list, (u32)h_tc[TC_NFIX],
            MODE == 0 ? ani_reparse : tree_reparse,
            [=] __device__(const AniPatch &p) {
                L.kind[p.line] = (u8)p.kind;
                if (MODE == 0) { L.m[p.line] = p.m; L.b[p.line] = p.b; }
                L.ql[p.line] = p.ql; L.tl[p.line] = p.tl;
            });
    const u32 n = (u32)n_ok;
    if (n == 0) return 0;
    *R = take_records<READER>(c, dl, L, n);
    *nt = intern_names(c, dl.text, tx, *R, n, tc, dl.d_cnt);
    return n;
}

// Genome of every sequence under `prefix`, as its rank among the sorted distinct genomes (*genomes): equal ranks <=> same
// genome, and min / max of two ranks orders a pair as the reference's (String, String) key does (main.rs:455-459).
static std::vector<u32> genome_ranks(const std::vector<std::string> &names, std::string (*prefix)(const std::string &),
                                     std::vector<std::string> *genomes) {
    std::vector<std::string> pre(names.size());
    for (size_t s = 0; s < names.size(); s++) pre[s] = prefix(names[s]);
    *genomes = pre;
    std::sort(genomes->begin(), genomes->end());
    genomes->erase(std::unique(genomes->begin(), genomes->end()), genomes->end());
    std::vector<u32> rank(names.size());
    for (size_t s = 0; s < names.size(); s++) rank[s] = (u32)(std::lower_bound(genomes->begin(), genomes->end(), pre[s]) - genomes->begin());
    return rank;
}

// method: SWG_ANI_ALL or SWG_ANI_NPERCENTILE (Orthogonal = the 1:1 filter first, then ALL; done by the caller).
static AniResult ani_device(swg_ctx *c, const swg_paf &hp, int method, double percentile, int sort) {
    cudaStream_t st = c->stream;
    LaunchCounter &lc = c->lc;
    Arena &A = c->io;
    AniResult res;
    const PafText tx(hp);
    const DevLines dl = load_lines(c, tx);
    if (hp.text_len == 0) return res;
    u32 *bsum = dl.bsum, *d_cnt = dl.d_cnt;
    u64 *tc = A.take<u64>(TC_COUNT);
    u64 h_tc[TC_COUNT];
    SWG_CUDA(cudaMemsetAsync(tc, 0, sizeof(u64) * TC_COUNT, st));
    TokCols R;
    NameTable nt;
    const u32 n = ani_records<0>(c, tx, dl, tc, &R, &nt);
    if (n == 0) return res;
    const u32 n_seq = nt.n_seq;
    std::vector<std::string> genomes;
    const std::vector<u32> seq_rank = genome_ranks(nt.names, paf_prefix_P, &genomes);
    const u32 nP = (u32)genomes.size();
    u32 *d_rank = A.take<u32>(n_seq);
    SWG_CUDA(cudaMemcpyAsync(d_rank, seq_rank.data(), (size_t)n_seq * 4, cudaMemcpyHostToDevice, st));
    // ---- inter-genome alignments, pair keys, sort keys -------------------------------------------------------
    u64 *pairkey = A.take<u64>(n);
    u64 *skey = A.take<u64>(n), *skey2 = A.take<u64>(n);
    u32 *sval = A.take<u32>(n), *sval2 = A.take<u32>(n);
    const u32 *qid = nt.qid, *tid = nt.tid;
    const u64 nP64 = nP;
    const bool npct = method == SWG_ANI_NPERCENTILE;
    {
        u64 *sk = skey;
        u32 *sv = sval;
        launch_for<t_ani_pairs>(n, st, lc, [=] __device__(u32 r) {
            const u32 a = d_rank[qid[r]], b2 = d_rank[tid[r]];
            const bool inter = a != b2; // main.rs:436-438
            pairkey[r] = inter ? (u64)min(a, b2) * nP64 + max(a, b2) : NONE64;
            u64 key = NONE64; // self comparisons sort behind everything
            bool isnan_ = false, nonint = false;
            if (inter && npct) {
                const double m = R.m[r], b = R.b[r];
                const double identity = __ddiv_rn(m, fmax(b, 1.0)); // main.rs:592
                double k = sort == SWG_NSORT_LENGTH ? b : sort == SWG_NSORT_IDENTITY ? identity : __dmul_rn(identity, fmax(log(b), 1.0));
                isnan_ = k != k;
                if (k == 0.0) k = 0.0; // -0.0 and +0.0 compare equal in partial_cmp
                key = score_desc_key(k);
                if (key == NONE64) key = NONE64 - 1;
                nonint = !(b >= 0.0 && b < 9007199254740992.0 && b == floor(b));
            }
            sk[r] = key;
            sv[r] = r;
            const u32 full = __activemask();
            const u32 c_inter = __popc(__ballot_sync(full, inter)), c_nan = __popc(__ballot_sync(full, isnan_)), c_non = __popc(__ballot_sync(full, nonint));
            if ((threadIdx.x & 31) == (u32)(__ffs(full) - 1)) {
                if (c_inter) atomicAdd((unsigned long long *)&tc[TC_INTER], (unsigned long long)c_inter);
                if (c_nan) atomicAdd((unsigned long long *)&tc[TC_NAN], (unsigned long long)c_nan);
                if (c_non) atomicAdd((unsigned long long *)&tc[TC_NONINT], (unsigned long long)c_non);
            }
        });
    }
    tok_read(c, tc, h_tc);
    const u32 n_inter = (u32)h_tc[TC_INTER];
    res.n_alignments = n_inter;
    if (n_inter == 0) return res; // main.rs:468-471 / :606-609
    if (h_tc[TC_NAN]) throw NanError{};
    // order[k] = record of the k-th alignment in the reference's accumulation order; the first `take` are used
    u32 take = n_inter;
    const u32 *order = nullptr; // nullptr: record order
    if (npct) {
        sort_pairs(c, skey, skey2, sval, sval2, n, 64); // stable: ties keep file order (Vec::sort_by is stable)
        order = sval;
        // total genome size: every distinct sequence of an inter-genome alignment once, with the length of its first appearance
        u64 *first = A.take<u64>(n_seq);
        u64 *seqlen = A.take<u64>(n_seq);
        SWG_CUDA(cudaMemsetAsync(first, 0xFF, sizeof(u64) * (size_t)n_seq, st));
        launch_for<t_ani_first>(n, st, lc, [=] __device__(u32 r) {
            if (pairkey[r] == NONE64) return;
            const u32 q = qid[r], t = tid[r];
            if (first[q] > 2ull * r) atomicMin((unsigned long long *)&first[q], 2ull * r);
            if (first[t] > 2ull * r + 1) atomicMin((unsigned long long *)&first[t], 2ull * r + 1);
        });
        launch_for<t_ani_sizes>(n_seq, st, lc, [=] __device__(u32 s) {
            const u64 f = first[s];
            seqlen[s] = f == NONE64 ? 0 : ((f & 1) ? R.tl[f >> 1] : R.ql[f >> 1]);
        });
        std::vector<u64> h_len(n_seq);
        SWG_CUDA(cudaMemcpyAsync(h_len.data(), seqlen, (size_t)n_seq * 8, cudaMemcpyDeviceToHost, st));
        SWG_CUDA(cudaStreamSynchronize(st));
        double total = 0.0;
        for (u32 s = 0; s < n_seq; s++) total += (double)h_len[s]; // main.rs:634 (a HashMap-order sum there; exact below 2^53)
        const double thr = total * (percentile / 100.0);           // main.rs:638
        // cumulative block length in sorted order, cut at the first alignment that reaches thr (inclusive)
        double *bsorted = A.take<double>(n_inter);
        {
            const u32 *ord = order;
            launch_for<t_ani_gather>(n_inter, st, lc, [=] __device__(u32 k) { bsorted[k] = R.b[ord[k]]; });
        }
        if (h_tc[TC_NONINT] == 0) {
            const u32 TILE = 1024;
            const u32 ntiles = cdiv(n_inter, TILE);
            u64 *tsum = A.take<u64>(ntiles);
            launch_for<t_ani_tiles>(ntiles, st, lc, [=] __device__(u32 t) {
                u64 s = 0;
                const u32 e = min((t + 1) * TILE, n_inter);
                for (u32 k = t * TILE; k < e; k++) s += (u64)bsorted[k];
                tsum[t] = s;
            });
            std::vector<u64> h_t(ntiles);
            SWG_CUDA(cudaMemcpyAsync(h_t.data(), tsum, (size_t)ntiles * 8, cudaMemcpyDeviceToHost, st));
            SWG_CUDA(cudaStreamSynchronize(st));
            unsigned __int128 cum = 0;
            bool exact = true;
            for (u32 t = 0; t < ntiles; t++) { cum += h_t[t]; if (cum >= ((unsigned __int128)1 << 53)) exact = false; }
            if (exact) {
                u64 before = 0;
                u32 t = 0;
                for (; t < ntiles; t++) {
                    if ((double)(before + h_t[t]) >= thr) break; // integers below 2^53: the f64 running sum of the reference is exact
                    before += h_t[t];
                }
                if (t < ntiles) {
                    const u32 k0 = t * TILE, cnt = std::min(TILE, n_inter - k0);
                    std::vector<double> hb(cnt);
                    SWG_CUDA(cudaMemcpyAsync(hb.data(), bsorted + k0, (size_t)cnt * 8, cudaMemcpyDeviceToHost, st));
                    SWG_CUDA(cudaStreamSynchronize(st));
                    double cumd = (double)before;
                    for (u32 k = 0; k < cnt; k++) {
                        cumd += hb[k];
                        if (cumd >= thr) { take = k0 + k + 1; break; }
                    }
                }
            } else take = 0; // fall through to the sequential walk
        }
        if (h_tc[TC_NONINT] != 0 || take == 0) { // non-integer block lengths: the rounding of the running sum is order dependent
            std::vector<double> hb(n_inter);
            SWG_CUDA(cudaMemcpyAsync(hb.data(), bsorted, (size_t)n_inter * 8, cudaMemcpyDeviceToHost, st));
            SWG_CUDA(cudaStreamSynchronize(st));
            double cumd = 0.0;
            take = n_inter;
            for (u32 k = 0; k < n_inter; k++) {
                cumd += hb[k];
                if (cumd >= thr) { take = k + 1; break; }
            }
        }
    }
    // ---- bring every pair's addends together, in order -----------------------------------------------------------
    const u32 n_items = npct ? take : n; // positions that take part in the pair sort (self comparisons carry a dead key)
    u64 *pk = A.take<u64>(n_items), *pk2 = A.take<u64>(n_items);
    u32 *pv = A.take<u32>(n_items), *pv2 = A.take<u32>(n_items);
    const int pbits = bits_for((u64)nP * nP) + 1;
    if (pbits > 63) throw RangeError{"too many genomes for the pair key"};
    const u64 dead = (1ull << pbits) - 1;
    {
        const u32 *ord = order;
        launch_for<t_ani_keys>(n_items, st, lc, [=] __device__(u32 k) {
            const u32 r = ord ? ord[k] : k;
            const u64 key = pairkey[r];
            pk[k] = key == NONE64 ? dead : key;
            pv[k] = r;
        });
    }
    sort_pairs(c, pk, pk2, pv, pv2, n_items, pbits);
    const u32 n_used = npct ? take : n_inter; // live keys sort first
    double *ms = A.take<double>(n_used), *bs = A.take<double>(n_used);
    u32 *seg_start = A.take<u32>(n_used);
    {
        const u64 *pkc = pk;
        const u32 *pvc = pv;
        scan_apply([=] __device__(u32 k) -> u32 { return (k == 0 || pkc[k] != pkc[k - 1]) ? 1u : 0u; },
                   [=] __device__(u32 k, u32 ex, u32 v) {
                       if (v) seg_start[ex] = k;
                       const u32 r = pvc[k];
                       ms[k] = R.m[r];
                       bs[k] = R.b[r];
                   },
                   n_used, bsum, d_cnt, st, lc);
    }
    const u32 n_pairs = read_u32(c, d_cnt);
    double *ani = A.take<double>(n_pairs);
    k_ani_pair_sums<<<cdiv(n_pairs, 128), 128, 0, st>>>(ms, bs, seg_start, n_pairs, n_used, ani);
    lc.n++;
    std::vector<double> h_ani(n_pairs);
    SWG_CUDA(cudaMemcpyAsync(h_ani.data(), ani, (size_t)n_pairs * 8, cudaMemcpyDeviceToHost, st));
    SWG_CUDA(cudaStreamSynchronize(st));
    for (double v : h_ani) if (v != v) throw NanError{};
    std::sort(h_ani.begin(), h_ani.end());
    const size_t mid = h_ani.size() / 2;
    res.ani50 = (h_ani.size() % 2 == 0 && h_ani.size() > 1) ? (h_ani[mid - 1] + h_ani[mid]) / 2.0 : h_ani[mid]; // main.rs:490-495
    res.n_pairs = n_pairs;
    return res;
}

// ---- tree sparsification of an existing PAF (`--sparsify tree:k[,f[,r]]`) --------------------------------------
//   tree_filter_device  <- apply_tree_filter_to_paf   (src/tree_filter.rs:205-283)
// Per genome pair (the P2 prefix rule) Σ matches / Σ block length over u64 columns — integers, so the sums are
// order-free: sort by pair, warp-segmented reduction, one atomic per (warp, pair).  The pair list (thousands) goes
// to the host, select_tree_pairs picks the k nearest / k farthest / hashed-random pairs, the flags come back, and
// the kept lines are assembled on the device in input order (write_device, verbatim lines).
struct t_tree_keys; struct t_tree_sums; struct t_tree_status; struct t_tree_pairout;
struct TreeResult { u64 n_kept = 0, n_selected = 0; };

static TreeResult tree_filter_device(swg_ctx *c, const swg_paf &hp, const char *out_path, u64 k_nearest, u64 k_farthest, double random_fraction) {
    cudaStream_t st = c->stream;
    LaunchCounter &lc = c->lc;
    Arena &A = c->io;
    TreeResult res;
    const PafText tx(hp);
    const DevLines dl = load_lines(c, tx);
    DevPaf dp;
    dp.text = dl.text;
    dp.text_len = tx.bytes;
    if (tx.bytes == 0) { write_device(c, dp, nullptr, nullptr, {out_path}); return res; }
    u32 *bsum = dl.bsum, *d_cnt = dl.d_cnt;
    u64 *tc = A.take<u64>(TC_COUNT);
    u64 h_tc[TC_COUNT];
    SWG_CUDA(cudaMemsetAsync(tc, 0, sizeof(u64) * TC_COUNT, st));
    TokCols R;
    NameTable nt;
    const u32 n = ani_records<1>(c, tx, dl, tc, &R, &nt);
    if (n == 0) { write_device(c, dp, nullptr, nullptr, {out_path}); return res; }
    const u32 n_seq = nt.n_seq;
    // genome of every sequence under extract_genome_prefix (tree_filter.rs:15-25, the P2 rule)
    std::vector<std::string> genomes;
    const std::vector<u32> seq_rank = genome_ranks(nt.names, paf_prefix_P2, &genomes);
    const u64 nG = genomes.size();
    u32 *d_rank = A.take<u32>(n_seq);
    SWG_CUDA(cudaMemcpyAsync(d_rank, seq_rank.data(), (size_t)n_seq * 4, cudaMemcpyHostToDevice, st));
    const int pbits = bits_for(nG * nG) + 1;
    if (pbits > 63) throw RangeError{"too many genomes for the pair key"};
    const u64 dead = (1ull << pbits) - 1;
    u64 *pk = A.take<u64>(n), *pk2 = A.take<u64>(n);
    u32 *pv = A.take<u32>(n), *pv2 = A.take<u32>(n);
    const u32 *qid = nt.qid, *tid = nt.tid;
    {
        u64 *k = pk;
        u32 *v = pv;
        launch_for<t_tree_keys>(n, st, lc, [=] __device__(u32 r) {
            const u32 a = d_rank[qid[r]], b = d_rank[tid[r]];
            const bool inter = a != b; // tree_filter.rs:46-48
            k[r] = inter ? (u64)min(a, b) * nG + max(a, b) : dead;
            v[r] = r;
            const u32 am = __activemask();
            const u32 cnt = __popc(__ballot_sync(am, inter));
            if (cnt && (threadIdx.x & 31) == (u32)(__ffs(am) - 1)) atomicAdd((unsigned long long *)&tc[TC_INTER], (unsigned long long)cnt);
        });
    }
    sort_pairs(c, pk, pk2, pv, pv2, n, pbits);
    tok_read(c, tc, h_tc);
    const u32 n_inter = (u32)h_tc[TC_INTER];
    u8 *status = A.take<u8>(n);
    u32 *chain = A.take<u32>(n);
    SWG_CUDA(cudaMemsetAsync(status, 0, n, st));
    SWG_CUDA(cudaMemsetAsync(chain, 0, sizeof(u32) * (size_t)n, st));
    dp.n = n;
    dp.rec = R;
    if (n_inter == 0) { write_device(c, dp, status, chain, {out_path}); return res; }
    u32 *gid = A.take<u32>(n_inter), *seg_start = A.take<u32>(n_inter);
    {
        const u64 *pkc = pk;
        scan_apply([=] __device__(u32 k) -> u32 { return (k == 0 || pkc[k] != pkc[k - 1]) ? 1u : 0u; },
                   [=] __device__(u32 k, u32 ex, u32 v) {
                       if (v) seg_start[ex] = k;
                       gid[k] = ex + v - 1;
                   },
                   n_inter, bsum, d_cnt, st, lc);
    }
    const u32 n_pairs = read_u32(c, d_cnt);
    u64 *sums = A.take<u64>(2 * (size_t)n_pairs), *pkeys = A.take<u64>(n_pairs);
    SWG_CUDA(cudaMemsetAsync(sums, 0, sizeof(u64) * 2 * (size_t)n_pairs, st));
    {
        const u32 *pvc = pv;
        const u64 *pkc = pk;
        launch_for<t_tree_sums>(n_inter, st, lc, [=] __device__(u32 k) {
            const u32 r = pvc[k], p = gid[k];
            u64 m = R.ql[r], b = R.tl[r];
            // runs of one pair are contiguous: segmented reduction towards the first lane of each run
            const u32 am = __activemask();
            const u32 run = __match_any_sync(am, p);
            const u32 lane = threadIdx.x & 31;
            for (u32 off = 1; off < 32; off <<= 1) {
                const u64 tm = __shfl_down_sync(am, m, off), tb = __shfl_down_sync(am, b, off);
                if (lane + off < 32 && ((run >> (lane + off)) & 1u)) { m += tm; b += tb; }
            }
            if (lane == (u32)(__ffs(run) - 1)) {
                atomicAdd((unsigned long long *)&sums[2 * (size_t)p], (unsigned long long)m);
                atomicAdd((unsigned long long *)&sums[2 * (size_t)p + 1], (unsigned long long)b);
            }
        });
        launch_for<t_tree_pairout>(n_pairs, st, lc, [=] __device__(u32 p) { pkeys[p] = pkc[seg_start[p]]; });
    }
    std::vector<u64> h_sums(2 * (size_t)n_pairs), h_keys(n_pairs);
    SWG_CUDA(cudaMemcpyAsync(h_sums.data(), sums, sizeof(u64) * 2 * (size_t)n_pairs, cudaMemcpyDeviceToHost, st));
    SWG_CUDA(cudaMemcpyAsync(h_keys.data(), pkeys, sizeof(u64) * (size_t)n_pairs, cudaMemcpyDeviceToHost, st));
    SWG_CUDA(cudaStreamSynchronize(st));
    std::vector<u32> lo(n_pairs), hi(n_pairs);
    std::vector<double> ident(n_pairs);
    for (u32 p = 0; p < n_pairs; p++) {
        lo[p] = (u32)(h_keys[p] / nG);
        hi[p] = (u32)(h_keys[p] % nG);
        const double tm = (double)h_sums[2 * (size_t)p], tb = (double)h_sums[2 * (size_t)p + 1]; // tree_filter.rs:58-59: f64 sums of integers, exact below 2^53
        ident[p] = tb > 0.0 ? tm / tb : 0.0;
    }
    bool has_nan = false;
    std::vector<uint8_t> sel = tree_select_pairs(genomes, lo, hi, ident, k_nearest, k_farthest, random_fraction, &has_nan);
    if (has_nan) throw NanError{};
    u8 *d_sel = A.take<u8>(n_pairs);
    SWG_CUDA(cudaMemcpyAsync(d_sel, sel.data(), n_pairs, cudaMemcpyHostToDevice, st));
    {
        const u32 *pvc = pv;
        launch_for<t_tree_status>(n_inter, st, lc, [=] __device__(u32 k) { status[pvc[k]] = d_sel[gid[k]] ? OUT_PLAIN : 0; });
    }
    SWG_CUDA(cudaStreamSynchronize(st)); // sel lives on this stack frame
    for (u32 p = 0; p < n_pairs; p++) res.n_selected += sel[p];
    write_device(c, dp, status, chain, {out_path});
    // kept lines: the records of the selected pairs
    {
        u32 *d_kept = d_cnt + 1;
        scan_apply([=] __device__(u32 r) -> u32 { return status[r] == OUT_PLAIN ? 1u : 0u; }, [] __device__(u32, u32, u32) {}, n, bsum, d_kept, st, lc);
        res.n_kept = read_u32(c, d_kept);
    }
    return res;
}

} // namespace swg

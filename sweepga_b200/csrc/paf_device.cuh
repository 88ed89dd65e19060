// paf_device.cuh — device front end: PAF text -> SoA on the GPU, and the tagged output assembled on the GPU.
// (SURVEY §8f rows 1 and 2: the callers immediately before and after the filter.)
//
//   tokenize_device  <- PafFilter::extract_metadata  (src/paf_filter.rs:292-376)
//                       + paf::parse_cigar_counts    (src/paf.rs:32-64)
//   write_device     <- write_filtered_output        (src/paf_filter.rs:1689-1726)
//
// The file is copied to HBM once.  Kernels:
//   1. newline scan (16 B per thread through the one-pass scan) -> line start offsets
//   2. k_tok_parse: one thread per line: split the first 11 fields, parse the integers, hash the two names, walk
//      the tags (dv:f: / cg:Z:, the later one wins)
//   3. k_tok_long: lines longer than SWG_TOK_LONG bytes (base-level CIGARs): one warp per line, the CIGAR is
//      counted byte-parallel
//   4. name interning: open-addressing table on the 64-bit name hash with the first appearance (2*record+side)
//      as value, ids = rank of the first appearance; every record then verifies its name bytes against the
//      representative, so a hash collision is detected (the call falls back to the host front end), never silent
//   5. output: per-record output length -> scan -> one warp per kept record copies the line and writes the tags
// Anything outside the plain grammar (numbers with more than 19 digits, inf/nan or long decimal dv values) is not
// guessed on the device: the line is listed and the host's reference-exact line parser (paf_parse_line) patches it.
//
// The three PAF readers on the device (this filter front end, and the ANI and tree readers of ani_device.cuh) share
// what is not their own policy: the line grammar (line_len_raw / strip_cr, name_field, u64_field, count_records /
// raise_maxlen), the counter block (TC_*) and line kinds (TK_*), the column list (TokCols, for_each_col) with
// take_cols / take_records, and the host patch step for the listed lines (patch_lines).  Each reader keeps its own
// columns and tags.
#pragma once

#include <atomic>
#include <thread>
#include <type_traits>

#include <fcntl.h>
#include <unistd.h>

namespace swg {

struct t_fixgather; struct t_patch; struct t_name_assign; struct t_out_bounds; struct t_name_salt; struct t_file_recs;

__constant__ double c_pow10[23] = {1e0,  1e1,  1e2,  1e3,  1e4,  1e5,  1e6,  1e7,  1e8,  1e9,  1e10, 1e11,
                                   1e12, 1e13, 1e14, 1e15, 1e16, 1e17, 1e18, 1e19, 1e20, 1e21, 1e22};

enum : u8 { TK_SKIP = 0, TK_OK = 1, TK_ERR_RANGE = 2, TK_ERR_ORDER = 3, TK_FIX = 4, TK_LONG = 5 };
enum { TC_OK = 0, TC_ERRLINE, TC_NFIX, TC_NLONG, TC_MAXLEN, TC_COLLISION, TC_DISTINCT, TC_TABLE_FULL, TC_INTER, TC_NAN, TC_NONINT, TC_COUNT };

struct TokCols { // per line, then per record; a reader has only the columns it uses (take_cols)
    u64 *off;
    u32 *len;
    u32 *qs, *qe, *ts, *te, *blen, *matches;
    double *identity;
    u8 *strand, *kind;
    u64 *qh, *th;
    u32 *qlen, *trel, *tlen;
    double *m, *b; // ANI: final matches, block length
    u64 *ql, *tl;  // ANI: sequence lengths (columns 2 and 7); tree: matches, block length (columns 10 and 11)
};

// The readers, as a mask of which of them use a column.
enum : u32 { RD_FILTER = 1, RD_ANI = 2, RD_TREE = 4 };

// Every column of TokCols once, with the readers that use it: f(readers, c.column...) for the same column of each c.
#pragma nv_exec_check_disable
template <class F, class... C> __host__ __device__ __forceinline__ void for_each_col(F &&f, C &...c) {
    constexpr u32 ALL = RD_FILTER | RD_ANI | RD_TREE;
    f(ALL, c.off...); f(RD_FILTER | RD_TREE, c.len...);
    f(RD_FILTER, c.qs...); f(RD_FILTER, c.qe...); f(RD_FILTER, c.ts...); f(RD_FILTER, c.te...);
    f(RD_FILTER, c.blen...); f(RD_FILTER, c.matches...); f(RD_FILTER, c.identity...); f(RD_FILTER, c.strand...);
    f(ALL, c.kind...); f(ALL, c.qh...); f(ALL, c.th...); f(ALL, c.qlen...); f(ALL, c.trel...); f(ALL, c.tlen...);
    f(RD_ANI, c.m...); f(RD_ANI, c.b...); f(RD_ANI | RD_TREE, c.ql...); f(RD_ANI | RD_TREE, c.tl...);
}

struct TokHead {
    u64 qs, qe, ts, te, mt, bl;
    u64 qh, th;
    u32 qlen, trel, tlen, tag_off;
    bool plus, fix;
};

__device__ __forceinline__ u64 name_hash_finish(u64 h, u32 len) {
    h ^= (u64)len * 0x9E3779B97F4A7C15ull;
    h ^= h >> 33; h *= 0xff51afd7ed558ccdULL; h ^= h >> 33; h *= 0xc4ceb9fe1a85ec53ULL; h ^= h >> 33;
    return h == NONE64 ? h - 1 : h;
}

// ---- the line grammar of every reader ------------------------------------------------------------
// Length of line l without its '\n', clamped: a line of 4 GiB still trips the host's longest-line check (front-end fallback).
__device__ __forceinline__ u32 line_len_raw(const u64 *__restrict__ line_start, u32 l) {
    return (u32)min(line_start[l + 1] - 1 - line_start[l], (u64)0xFFFFFFF0u);
}
__device__ __forceinline__ u32 strip_cr(const char *line, u32 len) { // BufRead::lines strips "\r\n"
    if (len > 0 && line[len - 1] == '\r') len--;
    return len;
}

// The name field that starts at a: FNV-1a over its bytes, finished with its length.  b: advanced to the end of the field.
__device__ __forceinline__ u64 name_field(const char *line, u32 a, u32 &b, u32 len) {
    u64 hh = 0xcbf29ce484222325ull;
    while (b < len) {
        const u8 ch = (u8)line[b];
        if (ch == '\t') break;
        hh = (hh ^ ch) * 0x100000001B3ull;
        b++;
    }
    return name_hash_finish(hh, b - a);
}

// str::parse::<u64>().unwrap_or(dflt) of the field that starts at a (paf_filter.rs:308-317).  More than 19 digits may or
// may not overflow u64: fix is set and the host decides.  b: advanced to the end of the field.
__device__ __forceinline__ u64 u64_field(const char *line, u32 a, u32 &b, u32 len, u64 dflt, bool &fix) {
    u64 v = 0;
    u32 nd = 0;
    bool bad = false;
    while (b < len) {
        const u8 ch = (u8)line[b];
        if (ch == '\t') break;
        if (!(b == a && ch == '+')) {
            const u32 d = (u32)ch - '0';
            if (d > 9) bad = true;
            else { if (nd < 19) v = v * 10 + d; nd++; }
        }
        b++;
    }
    if (bad || nd == 0) return dflt;
    if (nd > 19) fix = true;
    return v;
}

// End of a per-line parse kernel's block: the lines that became records (ok) are counted, the longest line raised.
__device__ __forceinline__ void count_records(bool ok, u64 *__restrict__ tc) {
    const u32 nok = __syncthreads_count(ok);
    if (threadIdx.x == 0 && nok) atomicAdd((unsigned long long *)&tc[TC_OK], (unsigned long long)nok);
}
__device__ __forceinline__ void raise_maxlen(u32 len, u64 *__restrict__ tc) {
    const u32 mx = __reduce_max_sync(0xFFFFFFFFu, len);
    if (lane_id() == 0 && mx > (u32)tc[TC_MAXLEN]) atomicMax((unsigned long long *)&tc[TC_MAXLEN], (unsigned long long)mx);
}

// First 11 fields of a line.  false: fewer than 11 fields (the line is skipped, paf_filter.rs:302-304).
__device__ __forceinline__ bool tok_parse_head(const char *__restrict__ line, u32 len, TokHead &h) {
    u32 a = 0;
    h.fix = false;
    h.plus = false;
    u64 num[6];
#pragma unroll 1
    for (int nf = 0; nf < 11; nf++) {
        u32 b = a;
        if (nf == 0 || nf == 5) {
            const u64 hh = name_field(line, a, b, len);
            if (nf == 0) { h.qh = hh; h.qlen = b - a; }
            else { h.th = hh; h.trel = a; h.tlen = b - a; }
        } else if (nf == 2 || nf == 3 || nf >= 7) {
            const u64 v = u64_field(line, a, b, len, nf == 10 ? 1 : 0, h.fix);
            const int slot = nf == 2 ? 0 : nf == 3 ? 1 : nf - 5; // 7,8,9,10 -> 2,3,4,5
            num[slot] = v;
        } else {
            if (nf == 4) h.plus = (a < len && line[a] == '+');
            while (b < len && line[b] != '\t') b++;
            if (nf == 4) h.plus = h.plus && (b - a == 1);
        }
        if (b >= len) { // no tab after this field
            if (nf < 10) return false;
            a = len + 1;
            break;
        }
        a = b + 1;
    }
    h.qs = num[0]; h.qe = num[1]; h.ts = num[2]; h.te = num[3]; h.mt = num[4]; h.bl = num[5];
    h.tag_off = a;
    return true;
}

// str::parse::<f64> for the plain decimal grammar.  0: Err (the tag is ignored), 1: ok, 2: leave it to the host
// (inf / nan, more than 19 significant digits, exponents outside the exactly representable powers of ten).
// With a mantissa < 2^53 and |exponent| <= 22 one IEEE operation on two exact operands is correctly rounded,
// which is what the reference's parser returns.
__device__ __forceinline__ int tok_parse_f64(const char *__restrict__ s, u32 len, double &out) {
    if (len == 0) return 0;
    if (len > 48) return 2;
    u32 i = 0;
    bool neg = false;
    if (s[0] == '+' || s[0] == '-') { neg = s[0] == '-'; i = 1; }
    if (i >= len) return 0;
    {
        const u8 c0 = (u8)s[i];
        if (!((c0 >= '0' && c0 <= '9') || c0 == '.')) {
            const u8 lc = c0 | 0x20;
            return (lc == 'i' || lc == 'n') ? 2 : 0;
        }
    }
    u64 m = 0;
    int nsig = 0, ndig = 0, frac = 0;
    bool toolong = false;
    while (i < len) {
        const u32 d = (u32)(u8)s[i] - '0';
        if (d > 9) break;
        ndig++;
        if (m != 0 || d != 0) { if (nsig < 19) { m = m * 10 + d; nsig++; } else toolong = true; }
        i++;
    }
    if (i < len && s[i] == '.') {
        i++;
        while (i < len) {
            const u32 d = (u32)(u8)s[i] - '0';
            if (d > 9) break;
            ndig++;
            frac++;
            if (m != 0 || d != 0) { if (nsig < 19) { m = m * 10 + d; nsig++; } else toolong = true; }
            i++;
        }
    }
    if (ndig == 0) return 0;
    int e = 0;
    bool ebig = false;
    if (i < len && (s[i] == 'e' || s[i] == 'E')) {
        i++;
        bool eneg = false;
        if (i < len && (s[i] == '+' || s[i] == '-')) { eneg = s[i] == '-'; i++; }
        int ne = 0;
        while (i < len) {
            const u32 d = (u32)(u8)s[i] - '0';
            if (d > 9) break;
            if (ne < 4) e = e * 10 + (int)d; else ebig = true;
            ne++;
            i++;
        }
        if (ne == 0) return 0;
        if (eneg) e = -e;
    }
    if (i != len) return 0;
    if (toolong || ebig) return 2;
    if (m == 0) { out = neg ? -0.0 : 0.0; return 1; }
    const int de = e - frac;
    if (m > (1ull << 53) || de < -22 || de > 22) return 2;
    double v = __ull2double_rn(m);
    v = de < 0 ? __ddiv_rn(v, c_pow10[-de]) : __dmul_rn(v, c_pow10[de]);
    out = neg ? -v : v;
    return 1;
}

struct TokResult {
    u64 exact;
    double identity;
    bool fix;
};

__device__ __forceinline__ void tok_store(const TokCols &L, u32 l, const TokHead &h, const TokResult &r, u32 *fix_list, u64 *tc, bool &ok_out) {
    const u64 LIM = 0xFFFFFFFFull;
    u8 kind;
    if (r.fix || h.fix) {
        kind = TK_FIX;
        fix_list[atomicAdd((unsigned long long *)&tc[TC_NFIX], 1ull)] = l;
    } else kind = TK_OK;
    // values beyond the u32 SoA / end < start: the record stays, with an impossible interval (same rule as paf_parse_line);
    // the filter raises SWG_ERR_RANGE only if it survives the stage-1 retain
    const bool over = h.qs > LIM || h.qe > LIM || h.ts > LIM || h.te > LIM || h.bl > LIM || r.exact > LIM;
    auto sat = [LIM](u64 v) { return (u32)(v > LIM ? LIM : v); };
    L.kind[l] = kind;
    L.qh[l] = h.qh; L.th[l] = h.th;
    L.qlen[l] = h.qlen; L.trel[l] = h.trel; L.tlen[l] = h.tlen;
    if (kind == TK_OK) {
        L.qs[l] = over ? 0xFFFFFFFFu : (u32)h.qs; L.qe[l] = over ? 0u : (u32)h.qe; L.ts[l] = sat(h.ts); L.te[l] = sat(h.te);
        L.blen[l] = sat(h.bl); L.matches[l] = sat(r.exact);
        L.identity[l] = r.identity;
        L.strand[l] = h.plus ? '+' : '-';
    }
    ok_out = kind == TK_OK;
}

// One thread per line.
__global__ void __launch_bounds__(256) k_tok_parse(const char *__restrict__ text, const u64 *__restrict__ line_start, u32 n_lines,
                                                   u32 long_thresh, TokCols L, u32 *__restrict__ long_list, u32 *__restrict__ fix_list,
                                                   u64 *__restrict__ tc) {
    const u32 l = blockIdx.x * blockDim.x + threadIdx.x;
    bool ok = false;
    u32 len = 0;
    if (l < n_lines) {
        const u64 s = line_start[l];
        const char *line = text + s;
        len = strip_cr(line, line_len_raw(line_start, l));
        L.off[l] = s;
        L.len[l] = len;
        if (len > long_thresh) {
            L.kind[l] = TK_LONG;
            long_list[atomicAdd((unsigned long long *)&tc[TC_NLONG], 1ull)] = l;
        } else {
            TokHead h;
            if (!tok_parse_head(line, len, h)) L.kind[l] = TK_SKIP;
            else {
                TokResult r;
                r.fix = false;
                r.exact = h.mt;
                const double bld = __ull2double_rn(h.bl > 1 ? h.bl : 1);
                r.identity = __ddiv_rn(__ull2double_rn(h.mt), bld);
                // tags from column 12 on, in order, the later one wins (paf_filter.rs:326-343)
                u32 a = h.tag_off;
                while (a <= len) {
                    u32 b = a;
                    int type = 0;
                    if (len - a >= 5 && line[a + 2] == ':' && line[a + 4] == ':') {
                        if (line[a] == 'd' && line[a + 1] == 'v' && line[a + 3] == 'f') type = 1;
                        else if (line[a] == 'c' && line[a + 1] == 'g' && line[a + 3] == 'Z') type = 2;
                    }
                    if (type == 2) {
                        // Σ of '=' run lengths (paf.rs:32-64); Err (tag ignored) on an empty or overflowing number
                        u64 m = 0, num = 0;
                        bool have = false, overflow = false, err = false;
                        b = a + 5;
                        while (b < len) {
                            const u8 ch = (u8)line[b];
                            if (ch == '\t') break;
                            const u32 d = (u32)ch - '0';
                            if (d <= 9) {
                                if (num > 1844674407370955161ull || (num == 1844674407370955161ull && d > 5)) overflow = true;
                                num = num * 10 + d;
                                have = true;
                            } else if (!err) {
                                if (!have || overflow) err = true;
                                else {
                                    if (ch == '=') m += num;
                                    num = 0;
                                    have = false;
                                }
                            }
                            b++;
                        }
                        if (!err && m > 0) { r.exact = m; r.identity = __ddiv_rn(__ull2double_rn(m), bld); }
                    } else {
                        while (b < len && line[b] != '\t') b++;
                        if (type == 1) {
                            double dv;
                            const int rc = tok_parse_f64(line + a + 5, b - a - 5, dv);
                            if (rc == 1) r.identity = __dsub_rn(1.0, dv);
                            else if (rc == 2) r.fix = true;
                        }
                    }
                    if (b >= len) break;
                    a = b + 1;
                }
                tok_store(L, l, h, r, fix_list, tc, ok);
            }
        }
    }
    count_records(ok, tc);
    raise_maxlen(len, tc);
}

// One warp per long line: lane 0 reads the head, the warp walks the tags 32 bytes at a time.
__global__ void __launch_bounds__(128) k_tok_long(const char *__restrict__ text, const u32 *__restrict__ long_list, u32 n_long, TokCols L,
                                                  u32 *__restrict__ fix_list, u64 *__restrict__ tc) {
    const u32 full = 0xFFFFFFFFu;
    const u32 lane = lane_id();
    for (u32 w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < n_long; w += (gridDim.x * blockDim.x) >> 5) {
        const u32 l = long_list[w];
        const char *line = text + L.off[l];
        const u32 len = L.len[l];
        TokHead h;
        int head_ok = 0;
        if (lane == 0) head_ok = tok_parse_head(line, len, h) ? 1 : 0;
        head_ok = __shfl_sync(full, head_ok, 0);
        if (!head_ok) {
            if (lane == 0) L.kind[l] = TK_SKIP;
            continue;
        }
        const u64 bl = __shfl_sync(full, h.bl, 0);
        const u64 mt = __shfl_sync(full, h.mt, 0);
        const double bld = __ull2double_rn(bl > 1 ? bl : 1);
        TokResult r;
        r.fix = false;
        r.exact = mt;
        r.identity = __ddiv_rn(__ull2double_rn(mt), bld);
        u32 a = __shfl_sync(full, h.tag_off, 0);
        while (a <= len) {
            int type = 0;
            if (len - a >= 5 && line[a + 2] == ':' && line[a + 4] == ':') { // uniform loads
                if (line[a] == 'd' && line[a + 1] == 'v' && line[a + 3] == 'f') type = 1;
                else if (line[a] == 'c' && line[a + 1] == 'g' && line[a + 3] == 'Z') type = 2;
            }
            // find the end of the field; a cg field is counted on the way
            u32 b = type ? a + 5 : a;
            u64 m = 0;
            bool err = false, punt = false;
            const u32 body = b;
            while (true) {
                const u32 p = b + lane;
                const u8 ch = p < len ? (u8)line[p] : (u8)'\t';
                const u32 tabs = __ballot_sync(full, ch == '\t');
                const u32 upto = tabs ? (u32)__ffs(tabs) - 1 : 32u; // bytes of this step that belong to the field
                if (type == 2 && lane < upto) {
                    const u32 d = (u32)ch - '0';
                    if (d > 9) { // an operation: the digit run before it is its length
                        u64 v = 0, scale = 1;
                        u32 k = 0;
                        u32 q = p;
                        while (q > body && k < 20) {
                            const u32 dd = (u32)(u8)line[q - 1] - '0';
                            if (dd > 9) break;
                            v += dd * scale;
                            scale *= 10;
                            q--;
                            k++;
                        }
                        if (k == 0) err = true;          // "".parse::<u64>() is Err
                        else if (k >= 20) punt = true;   // may overflow: host
                        else if (ch == '=') m += v;
                    }
                }
                if (tabs || b + 32 >= len) { b = min(b + upto, len); break; }
                b += 32;
            }
            if (type == 2) {
                // the reference stops at the first Err; everything after it is irrelevant, and so is the sum
                const bool any_err = __any_sync(full, err), any_punt = __any_sync(full, punt);
                u64 tot = m;
                for (int o = 16; o; o >>= 1) tot += __shfl_xor_sync(full, tot, o);
                if (any_punt) r.fix = true;
                else if (!any_err && tot > 0) { r.exact = tot; r.identity = __ddiv_rn(__ull2double_rn(tot), bld); }
            } else if (type == 1) {
                double dv = 0.0;
                int rc = 0;
                if (lane == 0) rc = tok_parse_f64(line + a + 5, b - a - 5, dv);
                rc = __shfl_sync(full, rc, 0);
                dv = __shfl_sync(full, dv, 0);
                if (rc == 1) r.identity = __dsub_rn(1.0, dv);
                else if (rc == 2) r.fix = true;
            }
            if (b >= len) break;
            a = b + 1;
        }
        if (lane == 0) {
            bool ok;
            tok_store(L, l, h, r, fix_list, tc, ok);
            if (ok) atomicAdd((unsigned long long *)&tc[TC_OK], 1ull);
        }
    }
}

// ---- name interning ------------------------------------------------------------------------------
// table: key = 64-bit name hash, value = min over records of (2*record + side): the first appearance
__global__ void __launch_bounds__(256) k_name_insert(const u64 *__restrict__ qh, const u64 *__restrict__ th, u32 n, u64 *hk, u64 *hfirst,
                                                     u32 hmask, u64 *__restrict__ tc) {
    const u32 r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
#pragma unroll 1
    for (int side = 0; side < 2; side++) {
        const u64 key = side ? th[r] : qh[r];
        const u64 order = 2ull * r + side;
        u32 s = (u32)(key >> 7) & hmask;
        for (u32 probe = 0; probe <= hmask; probe++) {
            u64 k = hk[s];
            if (k == NONE64) {
                k = atomicCAS((unsigned long long *)&hk[s], (unsigned long long)NONE64, (unsigned long long)key);
                if (k == NONE64) {
                    const u64 d = atomicAdd((unsigned long long *)&tc[TC_DISTINCT], 1ull);
                    if (2 * (d + 1) > (u64)hmask) tc[TC_TABLE_FULL] = 1; // keep the load factor below 1/2: the host retries with a larger table
                    k = key;
                }
            }
            if (k == key) {
                // values only decrease: a plain read that already shows an earlier appearance makes the atomic unnecessary
                if (hfirst[s] > order) atomicMin((unsigned long long *)&hfirst[s], (unsigned long long)order);
                break;
            }
            s = (s + 1) & hmask;
            // a table past half full is retried larger: stop probing it (once full, a missing key would walk every slot)
            if ((probe & 31) == 31 && *(volatile const u64 *)&tc[TC_TABLE_FULL]) return;
        }
        if (tc[TC_TABLE_FULL]) return;
    }
}

__device__ __forceinline__ u32 name_find(const u64 *__restrict__ hk, u32 hmask, u64 key) {
    u32 s = (u32)(key >> 7) & hmask;
    while (hk[s] != key) s = (s + 1) & hmask;
    return s;
}

// ids + byte verification against the representative (the record / side of the first appearance)
// file of union position o (a byte, or a record): the largest k < K with fstart[k] <= o
template <class T> __device__ __forceinline__ u32 file_at(const T *fstart, u32 K, T o) {
    u32 lo = 0, hi = K;
    while (hi - lo > 1) {
        const u32 mid = (lo + hi) >> 1;
        if (fstart[mid] <= o) lo = mid;
        else hi = mid;
    }
    return lo;
}

// A union of K > 1 files (fstart: their union byte offsets) gives every file its own namespace: the hashes are salted with
// the file, and a representative counts only when it lies in the same file, so a salted-hash collision of equal names in
// two files is reported, never merged.
__global__ void __launch_bounds__(256) k_name_lookup(const char *__restrict__ text, TokCols R, u32 n, const u64 *__restrict__ hk,
                                                     const u32 *__restrict__ id_of_slot, u32 hmask, const u64 *__restrict__ rep_off,
                                                     const u32 *__restrict__ rep_len, const u64 *__restrict__ fstart, u32 K,
                                                     u32 *__restrict__ qid, u32 *__restrict__ tid, u64 *__restrict__ tc) {
    const u32 r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    bool mismatch = false;
    const u32 file = K > 1 ? file_at<u64>(fstart, K, R.off[r]) : 0;
#pragma unroll 1
    for (int side = 0; side < 2; side++) {
        const u64 key = side ? R.th[r] : R.qh[r];
        const u32 id = id_of_slot[name_find(hk, hmask, key)];
        const u32 len = side ? R.tlen[r] : R.qlen[r];
        const char *mine = text + R.off[r] + (side ? R.trel[r] : 0);
        const char *rep = text + rep_off[id];
        if (len != rep_len[id] || (K > 1 && file_at<u64>(fstart, K, rep_off[id]) != file)) mismatch = true;
        else if (mine != rep)
            for (u32 j = 0; j < len; j++)
                if (mine[j] != rep[j]) { mismatch = true; break; }
        (side ? tid : qid)[r] = id;
    }
    if (mismatch) tc[TC_COLLISION] = 1;
}

// ---- output --------------------------------------------------------------------------------------
__device__ __forceinline__ u32 dec_digits(u32 v) {
    return v < 10 ? 1 : v < 100 ? 2 : v < 1000 ? 3 : v < 10000 ? 4 : v < 100000 ? 5 : v < 1000000 ? 6 : v < 10000000 ? 7 : v < 100000000 ? 8
           : v < 1000000000 ? 9 : 10;
}
constexpr u8 OUT_PLAIN = 4; // status value of write_device: the line as it is (tree filter), no tags
__device__ __forceinline__ u32 out_suffix_len(u8 s, u32 chain) {
    if (s == OUT_PLAIN) return 1;
    const u32 stl = s == 1 ? 8 : s == 2 ? 7 : 10; // scaffold / rescued / unassigned
    return (chain ? 12 + dec_digits(chain) : 0) + 6 + stl + 1;
}
// one warp per record of the window: line bytes, then "\tch:Z:chain_<k>" (if any), "\tst:Z:<status>", "\n"
__global__ void __launch_bounds__(256) k_out_copy(const char *__restrict__ text, const u64 *__restrict__ off, const u32 *__restrict__ len,
                                                  const u8 *__restrict__ status, const u32 *__restrict__ chain_id, u32 r0, u32 nrec,
                                                  const u32 *__restrict__ out_off, char *__restrict__ out) {
    const u32 w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (w >= nrec) return;
    const u32 o = out_off[w];
    if (o == NONE32) return;
    const u32 r = r0 + w, lane = lane_id();
    const char *src = text + off[r];
    char *dst = out + o;
    const u32 n = len[r];
    for (u32 j = lane; j < n; j += 32) dst[j] = src[j];
    dst += n;
    const u8 s = status[r];
    if (s == OUT_PLAIN) {
        if (lane == 0) dst[0] = '\n';
        return;
    }
    const u32 chain = chain_id[r];
    const u32 nd = chain ? dec_digits(chain) : 0, pre = chain ? 12 + nd : 0;
    const u32 stl = s == 1 ? 8 : s == 2 ? 7 : 10;
    const u32 total = pre + 6 + stl + 1;
    for (u32 j = lane; j < total; j += 32) {
        char ch;
        if (j < pre) {
            if (j < 12) ch = "\tch:Z:chain_"[j];
            else {
                u32 v = chain;
                for (u32 k = nd - 1 - (j - 12); k; k--) v /= 10;
                ch = (char)('0' + v % 10);
            }
        } else {
            const u32 k = j - pre;
            if (k < 6) ch = "\tst:Z:"[k];
            else if (k < 6 + stl) ch = (s == 1 ? "scaffold" : s == 2 ? "rescued" : "unassigned")[k - 6];
            else ch = '\n';
        }
        dst[j] = ch;
    }
}

__device__ __forceinline__ u32 nl_mask(u32 x) { // 0x80 in every byte of x that is '\n'
    const u32 y = x ^ 0x0A0A0A0Au;
    return ~(((y & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | y | 0x7F7F7F7Fu);
}

// ==================================================================================================
// host driver
// ==================================================================================================
// The text the device readers see: one file, or many laid end to end as one union (swg_filter_paf_batch).  File k starts at
// union byte start[k]; a non-empty file that does not end in '\n' is followed by one '\n' of the union, so every file ends a
// line and its last line parses and is written exactly as without the terminator.
struct PafText {
    std::vector<const swg_paf *> files;
    std::vector<u64> start; // K + 1 entries; start[K] = bytes
    u64 bytes = 0;
    u64 mem_budget = 0;     // a union of K > 1 files whose lines need more device memory than this is declined (GroupTooLarge)
    explicit PafText(std::vector<const swg_paf *> f) : files(std::move(f)), start(files.size() + 1) {
        for (size_t k = 0; k < files.size(); k++) {
            start[k] = bytes;
            bytes += files[k]->text_len + (pads(k) ? 1 : 0);
        }
        start[files.size()] = bytes;
    }
    explicit PafText(const swg_paf &p) : PafText(std::vector<const swg_paf *>{&p}) {}
    u32 K() const { return (u32)files.size(); }
    bool pads(size_t k) const { const swg_paf &p = *files[k]; return p.text_len && p.text[p.text_len - 1] != '\n'; }
    // the file that holds union byte o (o < bytes), and the host copy of that byte
    u32 file_of(u64 o) const { return (u32)(std::upper_bound(start.begin(), start.end() - 1, o) - start.begin()) - 1; }
    const char *host(u64 o) const { const u32 k = file_of(o); return files[k]->text + (o - start[k]); }
};

struct DevPaf {
    char *text = nullptr;
    u64 text_len = 0;
    u64 n_lines = 0;
    u32 n = 0;
    TokCols rec{};        // per record
    u32 *rank = nullptr;  // line of each record; nullptr when every line is a record (rank[r] == r)
    u32 *qid = nullptr, *tid = nullptr;
    u32 n_seq = 0;
    u32 *P = nullptr, *P2 = nullptr;
    std::vector<std::string> names;
    std::vector<u32> hP, hP2;
    // per file of the text (K + 1 entries): first record and first sequence id; rec_off: device copy of file_rec (K > 1)
    std::vector<u32> file_rec, file_seq;
    u32 *rec_off = nullptr;
    double ms_upload = 0, ms_tokenize = 0;
};

struct Patch { u32 line, qs, qe, ts, te, blen, matches; u32 kind_strand; double identity; }; // a line re-parsed by the host
struct FrontEndFallback { std::string why; }; // the device front end declines: the caller uses the host front end
struct GroupTooLarge {}; // a union of files has more lines than one call may hold: the caller splits it (nothing was written)

// Device memory a text of `bytes` bytes and `lines` lines needs through the front end, the filter and the writer: the text
// twice (c->io), per line the tokeniser's line and record columns (~170 B), status and chain (5 B), k_prefilter's reserve
// (400 B per record) and the writer's margin (48 B per record), plus the writer's 1 GiB window.
constexpr u64 PAF_MEM_PER_BYTE = 2, PAF_MEM_PER_LINE = 640;
static u64 paf_union_memory(u64 bytes, u64 lines) { return PAF_MEM_PER_BYTE * bytes + PAF_MEM_PER_LINE * lines + (1ull << 30); }

static void tok_read(swg_ctx *c, const u64 *d_tc, u64 *h) {
    SWG_CUDA(cudaMemcpyAsync(h, d_tc, sizeof(u64) * TC_COUNT, cudaMemcpyDeviceToHost, c->stream));
    SWG_CUDA(cudaStreamSynchronize(c->stream));
}

struct DevLines { // the text in HBM and the start offset of every line (line_start[n_lines] = one past the last terminator)
    char *text = nullptr;
    u64 *line_start = nullptr;
    u32 n_lines = 0;
    u32 *bsum = nullptr, *d_cnt = nullptr; // scan scratch sized for the word scan (>= any per-line scan), 4 counters
};

// Copies the text to the device (c->io, which is reset) and finds the line starts.  Events c->ev[0] / c->ev[1] bracket the
// upload: one column whose slices are the files (read with pread where a file is mapped) and the terminators the union adds.
static DevLines load_lines(swg_ctx *c, const PafText &tx) {
    static const char nl = '\n';
    const u64 B = tx.bytes;
    cudaStream_t st = c->stream;
    LaunchCounter &lc = c->lc;
    if (B >= (1ull << 36)) throw FrontEndFallback{"input larger than 64 GiB"};
    Arena &A = c->io;
    A.reserve((size_t)B * 2 + ((size_t)64 << 20));
    c->arena.reserve((size_t)64 << 20); // scratch of the small sorts
    DevLines dl;
    if (B == 0) return dl;
    cudaEvent_t e0 = c->ev[0], e1 = c->ev[1];
    char *text = A.take<char>(B + 64);
    dl.text = text;
    PinCol col{text, (size_t)B, {}};
    for (u32 k = 0; k < tx.K(); k++) {
        const swg_paf &p = *tx.files[k];
        if (p.text_len) col.segs.push_back(PinSeg{(char *)p.text, tx.start[k], p.text_len, p.fd});
        if (tx.pads(k)) col.segs.push_back(PinSeg{(char *)&nl, tx.start[k] + p.text_len, 1});
    }
    SWG_CUDA(cudaEventRecord(e0, st));
    SWG_CUDA(cudaMemsetAsync(text + (B & ~(u64)15), 0, 48, st));
    SWG_CUDA(cudaEventRecord(c->ev_copy[0], st));
    SWG_CUDA(cudaStreamWaitEvent(c->copy_stream, c->ev_copy[0], 0));
    staged_h2d_cols(c, std::vector<PinCol>{col});
    SWG_CUDA(cudaEventRecord(c->ev_copy[1], c->copy_stream));
    SWG_CUDA(cudaStreamWaitEvent(st, c->ev_copy[1], 0));
    SWG_CUDA(cudaEventRecord(e1, st));

    // ---- 1. line starts (the text ends in '\n': every line has its terminator) -------------------
    const u32 nw = (u32)((B + 15) / 16);
    u32 *bsum = A.take<u32>(scan_temp_u32(nw));
    u32 *d_cnt = A.take<u32>(4);
    const uint4 *words = reinterpret_cast<const uint4 *>(text);
    auto count_nl = [=] __device__(u32 w) -> u32 {
        const uint4 v = words[w];
        return __popc(nl_mask(v.x)) + __popc(nl_mask(v.y)) + __popc(nl_mask(v.z)) + __popc(nl_mask(v.w));
    };
    scan_apply(count_nl, [] __device__(u32, u32, u32) {}, nw, bsum, d_cnt, st, lc);
    const u32 n_lines = read_u32(c, d_cnt);
    if (tx.K() > 1 && (n_lines >= 0x7FFFFFF0u || (tx.mem_budget && paf_union_memory(B, n_lines) > tx.mem_budget))) throw GroupTooLarge{};
    if (n_lines >= 0x7FFFFFF0u) throw RangeError{"too many lines (must be < 2^31 per context)"};
    dl.n_lines = n_lines;
    if (n_lines > nw) bsum = A.take<u32>(scan_temp_u32(n_lines)); // lines shorter than 16 bytes on average: the per-line scans need more tiles
    dl.bsum = bsum;
    dl.d_cnt = d_cnt;
    u64 *line_start = A.take<u64>((size_t)n_lines + 2);
    dl.line_start = line_start;
    {
        const u64 first_last[2] = {0, B};
        SWG_CUDA(cudaMemcpyAsync(line_start, &first_last[0], 8, cudaMemcpyHostToDevice, st));
        SWG_CUDA(cudaMemcpyAsync(line_start + n_lines, &first_last[1], 8, cudaMemcpyHostToDevice, st));
        SWG_CUDA(cudaStreamSynchronize(st)); // first_last lives on this stack frame
    }
    scan_apply(count_nl,
               [=] __device__(u32 w, u32 ex, u32 v) {
                   if (!v) return;
                   const uint4 q = words[w];
                   const u32 x[4] = {q.x, q.y, q.z, q.w};
                   u32 k = ex + 1;
#pragma unroll
                   for (int j = 0; j < 4; j++) {
                       u32 m = nl_mask(x[j]);
                       while (m) {
                           const u32 byte = (__ffs(m) - 1) >> 3;
                           line_start[k++] = (u64)w * 16 + j * 4 + byte + 1;
                           m &= m - 1;
                       }
                   }
               },
               nw, bsum, d_cnt, st, lc);
    return dl;
}

// Columns for n lines or records: the ones READER uses (for_each_col), the others nullptr.
template <u32 READER> static TokCols take_cols(Arena &A, u32 n) {
    TokCols C{};
    for_each_col([&](u32 used, auto *&col) { col = (used & READER) ? A.take<std::remove_reference_t<decltype(*col)>>(n) : nullptr; }, C);
    return C;
}

// Records = the lines of kind TK_OK, in line order: L itself when every line is one, else the columns of L compacted into
// new ones.  rank (when not nullptr) then receives a column with the line of each record; it stays untouched otherwise.
template <u32 READER> static TokCols take_records(swg_ctx *c, const DevLines &dl, const TokCols &L, u32 n, u32 **rank = nullptr) {
    if (n == dl.n_lines) return L;
    const TokCols R = take_cols<READER>(c->io, std::max<u32>(n, 1));
    u32 *rk = rank ? (*rank = c->io.take<u32>(std::max<u32>(n, 1))) : nullptr;
    scan_apply([=] __device__(u32 l) -> u32 { return L.kind[l] == TK_OK ? 1u : 0u; },
               [=] __device__(u32 l, u32 r, u32 v) {
                   if (!v) return;
                   if (rk) rk[r] = l;
                   for_each_col([&](u32 used, auto *dst, auto *src) { if (used & READER) dst[r] = src[l]; }, R, L);
               },
               dl.n_lines, dl.bsum, dl.d_cnt, c->stream, c->lc);
    return R;
}

// The lines the device does not decide (fix_list, nfix entries) go to the host reader: reparse(line, len, p) fills the
// patch record p of one line (p.line is set) and says whether the line is a record; one kernel then applies every record
// with apply(p).  The host reads the same bytes as the device: from line_start, without a final '\r'.  Returns how many
// of the lines are records.
template <class P, class Apply>
static u32 patch_lines(swg_ctx *c, const PafText &tx, const DevLines &dl, const u32 *fix_list, u32 nfix,
                       bool (*reparse)(const char *line, size_t len, P &p), Apply apply) {
    cudaStream_t st = c->stream;
    std::vector<u32> lines(nfix);
    std::vector<u64> se(2 * (size_t)nfix);
    u64 *d_se = c->io.take<u64>(2 * (size_t)nfix);
    const u64 *ls = dl.line_start;
    launch_for<t_fixgather>(nfix, st, c->lc, [=] __device__(u32 i) { const u32 l = fix_list[i]; d_se[2 * i] = ls[l]; d_se[2 * i + 1] = ls[l + 1] - 1; });
    SWG_CUDA(cudaMemcpyAsync(lines.data(), fix_list, (size_t)nfix * 4, cudaMemcpyDeviceToHost, st));
    SWG_CUDA(cudaMemcpyAsync(se.data(), d_se, (size_t)nfix * 16, cudaMemcpyDeviceToHost, st));
    SWG_CUDA(cudaStreamSynchronize(st));
    std::vector<P> patches(nfix);
    u32 n_ok = 0;
    for (u32 i = 0; i < nfix; i++) {
        size_t len = (size_t)(se[2 * i + 1] - se[2 * i]);
        const char *line = tx.host(se[2 * i]);
        if (len > 0 && line[len - 1] == '\r') len--;
        patches[i].line = lines[i];
        if (reparse(line, len, patches[i])) n_ok++;
    }
    P *d_p = c->io.take<P>(nfix);
    SWG_CUDA(cudaMemcpyAsync(d_p, patches.data(), sizeof(P) * nfix, cudaMemcpyHostToDevice, st));
    launch_for<t_patch>(nfix, st, c->lc, [=] __device__(u32 i) { const P p = d_p[i]; apply(p); });
    SWG_CUDA(cudaStreamSynchronize(st)); // patches lives on this stack frame
    return n_ok;
}

struct NameTable { // result of intern_names
    u32 *qid = nullptr, *tid = nullptr;
    u32 n_seq = 0;
    std::vector<std::string> names;
    std::vector<u32> file_seq; // first id of every file of the text (K + 1 entries)
};

__device__ __forceinline__ u64 name_salt(u64 h, u32 file) { return file ? name_hash_finish(h ^ ((u64)file * 0xD6E8FEB86659FD93ull), 0) : h; }

// Names -> ids in first-appearance order (query before target within a record).  R needs off / qh / th / qlen / trel /
// tlen; tc is the TC_COUNT counter block, d_cnt 4 scratch counters.  Memory comes from c->io.  A text of K > 1 files
// (fstart: their union offsets on the device) gets one namespace per file: the ids are file-major, file k's ids are
// [file_seq[k], file_seq[k + 1]) in that file's own first-appearance order.
static NameTable intern_names(swg_ctx *c, const char *text, const PafText &tx, const TokCols &R, u32 n, u64 *tc, u32 *d_cnt,
                              const u64 *fstart = nullptr) {
    cudaStream_t st = c->stream;
    LaunchCounter &lc = c->lc;
    Arena &A = c->io;
    const u32 K = tx.K();
    u64 h_tc[TC_COUNT];
    NameTable nt;
    u32 hcap = 1u << 16;
    u64 *hk = nullptr, *hfirst = nullptr;
    u32 D = 0;
    SWG_CUDA(cudaMemsetAsync(tc + TC_COLLISION, 0, sizeof(u64), st));
    if (K > 1)
        launch_for<t_name_salt>(n, st, lc, [=] __device__(u32 r) {
            const u32 f = file_at<u64>(fstart, K, R.off[r]);
            R.qh[r] = name_salt(R.qh[r], f);
            R.th[r] = name_salt(R.th[r], f);
        });
    while (true) {
        hk = A.take<u64>(hcap);
        hfirst = A.take<u64>(hcap);
        SWG_CUDA(cudaMemsetAsync(hk, 0xFF, sizeof(u64) * hcap, st));
        SWG_CUDA(cudaMemsetAsync(hfirst, 0xFF, sizeof(u64) * hcap, st));
        SWG_CUDA(cudaMemsetAsync(tc + TC_DISTINCT, 0, 2 * sizeof(u64), st)); // TC_DISTINCT, TC_TABLE_FULL
        k_name_insert<<<cdiv(n, 256), 256, 0, st>>>(R.qh, R.th, n, hk, hfirst, hcap - 1, tc);
        lc.n++;
        tok_read(c, tc, h_tc);
        if (!h_tc[TC_TABLE_FULL]) { D = (u32)h_tc[TC_DISTINCT]; break; }
        if (hcap >= (1u << 31)) throw FrontEndFallback{"too many distinct sequence names for the device table"};
        hcap = hcap >= (1u << 27) ? hcap * 2 : hcap * 16;
    }
    // occupied slots ordered by first appearance
    u64 *sk = A.take<u64>(D), *sk2 = A.take<u64>(D);
    u32 *sv = A.take<u32>(D), *sv2 = A.take<u32>(D);
    u32 *bsum2 = A.take<u32>(scan_temp_u32(hcap));
    scan_apply([=] __device__(u32 s) -> u32 { return hk[s] != NONE64 ? 1u : 0u; },
               [=] __device__(u32 s, u32 ex, u32 v) { if (v) { sk[ex] = hfirst[s]; sv[ex] = s; } }, hcap, bsum2, d_cnt, st, lc);
    sort_pairs(c, sk, sk2, sv, sv2, D, bits_for(2ull * n + 1));
    u32 *id_of_slot = A.take<u32>(hcap);
    u64 *rep_off = A.take<u64>(D);
    u32 *rep_len = A.take<u32>(D);
    {
        const u64 *skc = sk;
        const u32 *svc = sv;
        launch_for<t_name_assign>(D, st, lc, [=] __device__(u32 j) {
            id_of_slot[svc[j]] = j;
            const u64 order = skc[j];
            const u32 r = (u32)(order >> 1);
            const bool side = order & 1;
            rep_off[j] = R.off[r] + (side ? R.trel[r] : 0);
            rep_len[j] = side ? R.tlen[r] : R.qlen[r];
        });
    }
    nt.qid = A.take<u32>(n);
    nt.tid = A.take<u32>(n);
    k_name_lookup<<<cdiv(n, 256), 256, 0, st>>>(text, R, n, hk, id_of_slot, hcap - 1, rep_off, rep_len, fstart, K, nt.qid, nt.tid, tc);
    lc.n++;
    std::vector<u64> h_off(D);
    std::vector<u32> h_len(D);
    SWG_CUDA(cudaMemcpyAsync(h_off.data(), rep_off, (size_t)D * 8, cudaMemcpyDeviceToHost, st));
    SWG_CUDA(cudaMemcpyAsync(h_len.data(), rep_len, (size_t)D * 4, cudaMemcpyDeviceToHost, st));
    tok_read(c, tc, h_tc);
    if (h_tc[TC_COLLISION]) throw FrontEndFallback{"64-bit name hash collision"};
    nt.n_seq = D;
    nt.names.resize(D);
    nt.file_seq.assign(K + 1, 0);
    for (u32 j = 0; j < D; j++) {
        const u32 f = K > 1 ? tx.file_of(h_off[j]) : 0;
        nt.names[j].assign(tx.files[f]->text + (h_off[j] - tx.start[f]), h_len[j]);
        nt.file_seq[f + 1]++;
    }
    for (u32 k = 0; k < K; k++) nt.file_seq[k + 1] += nt.file_seq[k];
    return nt;
}

// Tokenise the text on the device.  All device memory comes from c->io and stays valid until the next front-end call.
static void tokenize_device(swg_ctx *c, const PafText &tx, DevPaf &dp) {
    const u32 long_thresh = c->knobs.tok_long;
    const u64 B = tx.bytes;
    const u32 K = tx.K();
    cudaStream_t st = c->stream;
    LaunchCounter &lc = c->lc;
    Arena &A = c->io;
    dp = DevPaf();
    dp.text_len = B;
    dp.file_rec.assign(K + 1, 0);
    dp.file_seq.assign(K + 1, 0);
    const DevLines dl = load_lines(c, tx);
    if (B == 0) return;
    cudaEvent_t e0 = c->ev[0], e1 = c->ev[1], e2 = c->ev[2];
    char *text = dl.text;
    dp.text = text;
    const u32 n_lines = dl.n_lines;
    dp.n_lines = n_lines;
    const u64 *line_start = dl.line_start;
    u32 *d_cnt = dl.d_cnt;

    // ---- 2./3. per-line parse --------------------------------------------------------------------
    const TokCols L = take_cols<RD_FILTER>(A, n_lines);
    u32 *long_list = A.take<u32>(n_lines), *fix_list = A.take<u32>(n_lines);
    u64 *tc = A.take<u64>(TC_COUNT);
    u64 h_tc[TC_COUNT];
    SWG_CUDA(cudaMemsetAsync(tc, 0, sizeof(u64) * TC_COUNT, st));
    SWG_CUDA(cudaMemsetAsync(tc + TC_ERRLINE, 0xFF, sizeof(u64), st));
    k_tok_parse<<<cdiv(n_lines, 256), 256, 0, st>>>(text, line_start, n_lines, long_thresh, L, long_list, fix_list, tc);
    lc.n++;
    tok_read(c, tc, h_tc);
    if (h_tc[TC_NLONG]) {
        const u32 n_long = (u32)h_tc[TC_NLONG];
        k_tok_long<<<std::min<u32>(cdiv((u64)n_long * 32, 128), (u32)c->sm_count * 16), 128, 0, st>>>(text, long_list, n_long, L, fix_list, tc);
        lc.n++;
        tok_read(c, tc, h_tc);
    }
    if (h_tc[TC_MAXLEN] > ((u64)256 << 20)) throw FrontEndFallback{"a line longer than 256 MiB"};
    c->tok_maxlen = (u32)h_tc[TC_MAXLEN];
    u64 n_ok = h_tc[TC_OK];
    // ---- lines the device does not decide: the host's reference-exact parser patches them -----------
    if (h_tc[TC_NFIX])
        n_ok += patch_lines<Patch>(
            c, tx, dl, fix_list, (u32)h_tc[TC_NFIX],
            [](const char *line, size_t len, Patch &p) {
                PafLine pl;
                const bool ok = paf_parse_line(line, len, &pl) != PafLine::SKIP; // range / order problems ride along as impossible intervals
                p.qs = pl.qs; p.qe = pl.qe; p.ts = pl.ts; p.te = pl.te; p.blen = pl.blen; p.matches = pl.matches;
                p.identity = pl.identity;
                p.kind_strand = (u32)(ok ? TK_OK : TK_SKIP) | ((u32)pl.strand << 8);
                return ok;
            },
            [=] __device__(const Patch &p) {
                const u32 l = p.line;
                L.kind[l] = (u8)(p.kind_strand & 0xFF);
                L.qs[l] = p.qs; L.qe[l] = p.qe; L.ts[l] = p.ts; L.te[l] = p.te; L.blen[l] = p.blen; L.matches[l] = p.matches;
                L.identity[l] = p.identity;
                L.strand[l] = (u8)(p.kind_strand >> 8);
            });

    // ---- records = lines that parsed (compaction only when some line did not) ----------------------
    const u32 n = (u32)n_ok;
    dp.n = n;
    const TokCols R = take_records<RD_FILTER>(c, dl, L, n, &dp.rank);
    dp.rec = R;
    if (n == 0) { SWG_CUDA(cudaStreamSynchronize(st)); return; }

    // ---- first record of every file: its first line (the line that starts at its union offset), or the first record at or
    // after that line when lines were dropped ----------------------------------------------------------------------------
    u64 *fstart = nullptr;
    if (K > 1) {
        fstart = A.take<u64>(K + 1);
        dp.rec_off = A.take<u32>(K + 1);
        SWG_CUDA(cudaMemcpyAsync(fstart, tx.start.data(), sizeof(u64) * (K + 1), cudaMemcpyHostToDevice, st));
        u32 *rec_off = dp.rec_off;
        const u32 *rank = dp.rank;
        launch_for<t_file_recs>(K + 1, st, lc, [=] __device__(u32 k) {
            u32 lo = 0, hi = n_lines;
            while (lo < hi) { const u32 mid = (lo + hi) >> 1; if (line_start[mid] < fstart[k]) lo = mid + 1; else hi = mid; }
            const u32 line = lo;
            if (rank) {
                lo = 0; hi = n;
                while (lo < hi) { const u32 mid = (lo + hi) >> 1; if (rank[mid] < line) lo = mid + 1; else hi = mid; }
            }
            rec_off[k] = lo;
        });
        SWG_CUDA(cudaMemcpyAsync(dp.file_rec.data(), rec_off, sizeof(u32) * (K + 1), cudaMemcpyDeviceToHost, st));
    } else dp.file_rec[1] = n;

    // ---- 4. names -> ids in first-appearance order ------------------------------------------------
    {
        NameTable nt = intern_names(c, text, tx, R, n, tc, d_cnt, fstart);
        dp.qid = nt.qid;
        dp.tid = nt.tid;
        dp.n_seq = nt.n_seq;
        dp.names.swap(nt.names);
        dp.file_seq.swap(nt.file_seq);
    }
    const u32 D = dp.n_seq;
    // genome prefixes P and P2 per file, the ids of file k shifted by the genomes of the files before it
    if (K == 1) paf_prefix_ids(dp.names, &dp.hP, &dp.hP2);
    else {
        dp.hP.resize(D);
        dp.hP2.resize(D);
        u32 goff = 0;
        std::vector<u32> p, p2;
        for (u32 k = 0; k < K; k++) {
            const u32 a = dp.file_seq[k], b = dp.file_seq[k + 1];
            if (a == b) continue;
            paf_prefix_ids(std::vector<std::string>(dp.names.begin() + a, dp.names.begin() + b), &p, &p2);
            u32 mx = 0;
            for (u32 j = 0; j < b - a; j++) {
                dp.hP[a + j] = p[j] + goff;
                dp.hP2[a + j] = p2[j] + goff;
                mx = std::max(mx, std::max(p[j], p2[j]));
            }
            goff += mx + 1;
        }
    }
    dp.P = A.take<u32>(D);
    dp.P2 = A.take<u32>(D);
    SWG_CUDA(cudaMemcpyAsync(dp.P, dp.hP.data(), (size_t)D * 4, cudaMemcpyHostToDevice, st));
    SWG_CUDA(cudaMemcpyAsync(dp.P2, dp.hP2.data(), (size_t)D * 4, cudaMemcpyHostToDevice, st));
    SWG_CUDA(cudaEventRecord(e2, st));
    SWG_CUDA(cudaStreamSynchronize(st));
    float m0 = 0, m1 = 0;
    cudaEventElapsedTime(&m0, e0, e1);
    cudaEventElapsedTime(&m1, e1, e2);
    dp.ms_upload = m0;
    dp.ms_tokenize = m1;
}

static DevIn devin_of(const DevPaf &dp) {
    DevIn d;
    d.qid = dp.qid; d.tid = dp.tid; d.qs = dp.rec.qs; d.qe = dp.rec.qe; d.ts = dp.rec.ts; d.te = dp.rec.te;
    d.blen = dp.rec.blen; d.matches = dp.rec.matches; d.identity = dp.rec.identity; d.strand = dp.rec.strand;
    d.score = nullptr; d.P = dp.P; d.P2 = dp.P2; d.n = dp.n; d.n_seq = dp.n_seq;
    return d;
}

// Tagged output, assembled on the device window by window (1 GiB of input text per window keeps every offset in u32),
// copied back through the pinned pieces and written with pwrite()s.  out_paths: one per file of the text (dp.file_rec; a
// DevPaf without it is one file).  The outputs of the files are consecutive ranges of the union's output: a piece goes to
// every file it overlaps, at its output position minus the file's base (the output position of the file's first record,
// taken from the window's scan once the window that holds that record is assembled).
static void write_device(swg_ctx *c, const DevPaf &dp, const u8 *status, const u32 *chain_id, const std::vector<const char *> &out_paths) {
    const bool trace = c->knobs.stage_timing;
    const auto t_begin = std::chrono::steady_clock::now();
    auto lap = [&](const char *what) {
        if (trace) fprintf(stderr, "[swg write] %s at %.1f ms\n", what, std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count());
    };
    const u32 K = (u32)out_paths.size();
    struct Closer { std::vector<int> fd; ~Closer() { for (int f : fd) if (f >= 0) close(f); } } closer{std::vector<int>(K, -1)};
    std::vector<int> &fds = closer.fd;
    for (u32 k = 0; k < K; k++) {
        fds[k] = open(out_paths[k], O_WRONLY | O_CREAT | O_TRUNC, 0644);
        if (fds[k] < 0) throw IoError{std::string("cannot create ") + out_paths[k]};
    }
    lap("open");
    const u32 n = dp.n;
    if (n == 0) return;
    ensure_pinned(c);
    cudaStream_t st = c->stream;
    LaunchCounter &lc = c->lc;
    Arena &A = c->arena; // continues behind run_filter's allocations (the chain keys of the last call stay readable)
    const u64 W = (u64)1 << 30;
    const u32 nwin = (u32)(dp.text_len / W) + 1;
    u32 *d_bounds = A.take<u32>(nwin + 1);
    {
        const u64 *off = dp.rec.off;
        launch_for<t_out_bounds>(nwin + 1, st, lc, [=] __device__(u32 k) {
            const u64 target = (u64)k * W;
            u32 lo = 0, hi = n;
            while (lo < hi) { const u32 mid = (lo + hi) >> 1; if (off[mid] < target) lo = mid + 1; else hi = mid; }
            d_bounds[k] = k == nwin ? n : lo;
        });
    }
    std::vector<u32> bounds(nwin + 1);
    SWG_CUDA(cudaMemcpyAsync(bounds.data(), d_bounds, (nwin + 1) * 4, cudaMemcpyDeviceToHost, st));
    SWG_CUDA(cudaStreamSynchronize(st));
    u32 max_rec = 0;
    for (u32 k = 0; k < nwin; k++) max_rec = std::max(max_rec, bounds[k + 1] - bounds[k]);
    u32 *out_off = A.take<u32>(max_rec);
    u32 *bsum = A.take<u32>(scan_temp_u32(max_rec));
    u32 *d_tot = A.take<u32>(4);
    char *out = A.take<char>(std::min<u64>(W, dp.text_len) + c->tok_maxlen + (u64)48 * max_rec + 256);
    const u32 *len = dp.rec.len;
    // the files with records, in order, and their output bases (UINT64_MAX until known)
    const std::vector<u32> frec = dp.file_rec.empty() ? std::vector<u32>{0, n} : dp.file_rec;
    std::vector<u32> live;
    for (u32 k = 0; k < K; k++)
        if (frec[k] < frec[k + 1]) live.push_back(k);
    std::vector<u64> live_base(live.size(), UINT64_MAX);
    std::vector<u32> h_base(K);
    u32 *d_base = K > 1 ? A.take<u32>(K) : nullptr;
    const u32 *rec_off = dp.rec_off;
    size_t known = 0; // live files whose base is known
    std::atomic<int> failed{0}; // 1: CUDA, 2: write
    std::atomic<u32> bad_file{0};
    u64 file_off = 0;
    for (u32 k = 0; k < nwin && !failed.load(); k++) {
        const u32 r0 = bounds[k], nrec = bounds[k + 1] - bounds[k];
        if (nrec == 0) continue;
        scan_apply([=] __device__(u32 w) -> u32 {
                       const u8 s = status[r0 + w];
                       return (s == 0 || s > OUT_PLAIN) ? 0u : len[r0 + w] + out_suffix_len(s, chain_id[r0 + w]);
                   },
                   [=] __device__(u32 w, u32 ex, u32 v) {
                       out_off[w] = v ? ex : NONE32;
                       if (K > 1) {
                           const u32 r = r0 + w, f = file_at<u32>(rec_off, K, r);
                           if (rec_off[f] == r) d_base[f] = ex;
                       }
                   },
                   nrec, bsum, d_tot, st, lc);
        k_out_copy<<<cdiv((u64)nrec * 32, 256), 256, 0, st>>>(dp.text, dp.rec.off, len, status, chain_id, r0, nrec, out_off, out);
        lc.n++;
        size_t now = known;
        while (now < live.size() && frec[live[now]] < r0 + nrec) now++;
        if (K > 1 && now > known)
            SWG_CUDA(cudaMemcpyAsync(h_base.data() + live[known], d_base + live[known], sizeof(u32) * (live[now - 1] + 1 - live[known]),
                                     cudaMemcpyDeviceToHost, st));
        const u32 total = read_u32(c, d_tot); // synchronises: the window is assembled
        for (; known < now; known++) live_base[known] = file_off + (K > 1 ? h_base[live[known]] : 0);
        lap("window assembled");
        // device -> pinned piece -> pwrite at its file offsets, one worker per piece buffer
        const size_t npieces = ((size_t)total + PIN_PIECE - 1) / PIN_PIECE;
        std::atomic<size_t> next{0};
        auto worker = [&](int t) {
            cudaSetDevice(c->device);
            while (!failed.load()) {
                const size_t p = next.fetch_add(1);
                if (p >= npieces) break;
                const size_t o = p * PIN_PIECE, l = std::min(PIN_PIECE, (size_t)total - o);
                if (cudaMemcpyAsync(c->pin[t], out + o, l, cudaMemcpyDeviceToHost, c->copy_stream) != cudaSuccess ||
                    cudaEventRecord(c->pin_ev[t], c->copy_stream) != cudaSuccess || cudaEventSynchronize(c->pin_ev[t]) != cudaSuccess) {
                    failed = 1;
                    break;
                }
                const u64 g0 = file_off + o, g1 = g0 + l;
                size_t i = (size_t)(std::upper_bound(live_base.begin(), live_base.end(), g0) - live_base.begin()) - 1;
                for (u64 g = g0; g < g1 && !failed.load(); i++) {
                    const u64 stop = std::min(g1, i + 1 < live_base.size() ? live_base[i + 1] : UINT64_MAX);
                    size_t done = 0;
                    while (g + done < stop) {
                        const ssize_t w = pwrite(fds[live[i]], c->pin[t] + (g - g0) + done, stop - g - done, (off_t)(g - live_base[i] + done));
                        if (w <= 0) { bad_file = live[i]; failed = 2; break; }
                        done += (size_t)w;
                    }
                    g = stop;
                }
            }
        };
        std::vector<std::thread> th;
        const int nt = (int)std::min<size_t>(PIN_COUNT, npieces);
        for (int t = 1; t < nt; t++) th.emplace_back(worker, t);
        if (nt > 0) worker(0);
        for (auto &t : th) t.join();
        file_off += total;
        lap("window written");
    }
    bool closed = true;
    for (u32 k = 0; k < K; k++) {
        if (close(fds[k]) != 0 && closed) { closed = false; bad_file = k; }
        fds[k] = -1;
    }
    lap("closed");
    if (failed.load() == 1) { cudaGetLastError(); throw CudaError{cudaErrorUnknown, __FILE__, __LINE__}; }
    if (failed.load() == 2 || !closed) throw IoError{std::string("write to ") + out_paths[bad_file.load()] + " failed"};
}

} // namespace swg
